#!/usr/bin/env python
"""bench.py - throughput of the UNet training / sampling hot path on B200.

    python bench.py --gpus N --steps K --warmup W            # this repo (libfdx kernels)
    python bench.py --impl reference --gpus N --steps K ...  # CPU reference arm (oracle on host cores)

A "step" is one data-parallel training step of the EDM UNet (noise-add -> UNet fwd -> weighted
L2 -> UNet bwd -> bucketed NCCL grad all-reduce overlapped with bwd -> AdamW + EMA) on a synthetic batch.
The headline keys are BASELINE.json configs[1] (unconditional EDM UNet 64x64x3, bf16, batch 256 per GPU);
the same default run covers the rest of the metric ("@64^2 & 256^2"): `sample` = Euler 50 steps at 64^2,
`train_256` = configs[2] (EDM UNet 256^2 with self-attention, B = 64 per GPU = 512 over 8 GPUs),
`sample_256_heun` = configs[4] (Heun 18/50/100 steps, B = 32 per GPU, replicas), `sample_256_text_cfg` =
configs[3] (text cross-attention, CFG Euler-ancestral 30 steps, B = 64).  Prints ONE JSON line.
Every timed training loop runs --steps steps.

    python bench.py ... --dump-outputs DIR   # also write what the timed path computed as DIR/<name>.npy

The inputs are seeded, so two builds run with the same arguments can be compared output for output: per training
workload the loss, parameters, EMA parameters and Adam moments after the last timed step; per sampler run the
images it returned.
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

FWD_GFLOP = {  # algorithmic forward GFLOP per image (BASELINE.md $2)
    ("c2", 64): 18.17, ("c3", 256): 300.83, ("c5", 256): 300.83, ("c4", 256): 298.03,
}
WORKLOADS = {
    # name: (resolution, per-GPU batch, attention configs, description)
    "c2": (64, 256, (None, None, None, None), "EDM UNet 64x64x3 bf16 B=256/GPU (BASELINE configs[1])"),
    "c3": (256, 64, (None, None, None, {"heads": 8}), "EDM UNet 256x256x3 self-attn bf16 B=64/GPU (configs[2])"),
    # sampling-only workloads (python bench.py --workload c4|c5): value = denoise steps / s
    "c4": (256, 64, (None, {"heads": 8}, {"heads": 8}, {"heads": 8}),
           "text-cond UNet 256x256x3 (frozen random 77x768 text emb), CFG g=3, Euler-ancestral 30 steps, B=64 (configs[3])"),
    "c5": (256, 32, (None, None, None, {"heads": 8}),
           "EDM UNet 256x256x3 self-attn, Heun 18/50/100 steps, B=32/GPU (configs[4])"),
}


def usable_cores() -> int:
    """Host cores this process may actually use: affinity mask capped by the cgroup CPU quota
    (os.cpu_count() reports the whole host inside a container and oversubscribes the thread pool)."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:  # noqa: BLE001
        n = os.cpu_count() or 1
    try:
        q = open("/sys/fs/cgroup/cpu.max").read().split()
        if q[0] != "max":
            n = min(n, max(1, int(int(q[0]) / int(q[1]))))
    except Exception:  # noqa: BLE001
        try:
            quota = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            period = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if quota > 0:
                n = min(n, max(1, quota // period))
        except Exception:  # noqa: BLE001
            pass
    return max(1, min(n, 64))


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("hbm_gbs", 6650.0), d.get("bf16_tflops", 1590.0), d.get("bf16_tflops_sustained", 1400.0), "measured"
    return 6650.0, 1590.0, 1400.0, "fallback"


_JSON_OUT = None


def claim_stdout():
    """Keep stdout for the ONE JSON line: everything else any library prints there (NCCL's version banner,
    for one) is sent to stderr for the rest of the run."""
    global _JSON_OUT
    if _JSON_OUT is None:
        sys.stdout.flush()
        _JSON_OUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(obj) -> None:
    out = _JSON_OUT if _JSON_OUT is not None else sys.stdout
    out.write(json.dumps(obj) + "\n")
    out.flush()


_OUTPUTS = None                 # name -> float32 host array, collected on rank 0 when --dump-outputs is given
OUTPUT_MAX_ELEMS = 1 << 20      # per array; 13 arrays in the default run stay under OUTPUT_MAX_BYTES
OUTPUT_MAX_BYTES = 64 << 20


def keep_output(name: str, t) -> None:
    """Record `t` for --dump-outputs as a float32 host copy; above OUTPUT_MAX_ELEMS elements, a sample at
    fixed seeded indices (the same indices in every run for the same size)."""
    if _OUTPUTS is None:
        return
    import numpy as np
    a = t.detach().float().cpu().numpy()
    if a.size > OUTPUT_MAX_ELEMS:
        a = a.reshape(-1)[np.sort(np.random.default_rng(0).integers(0, a.size, OUTPUT_MAX_ELEMS))]
    _OUTPUTS[name] = a


def write_outputs(directory: str) -> None:
    import numpy as np
    total = sum(a.nbytes for a in _OUTPUTS.values())
    if total > OUTPUT_MAX_BYTES:
        raise RuntimeError(f"--dump-outputs: {total} bytes exceed the {OUTPUT_MAX_BYTES}-byte limit")
    os.makedirs(directory, exist_ok=True)
    for name, a in _OUTPUTS.items():
        np.save(os.path.join(directory, name + ".npy"), a)


def roofline_traffic(workload: str, batch: int) -> dict:
    """DRAM bytes the tensor-core engine moved in one step, from the committed ncu pass (profiles/) of the
    same workload; null when no capture exists for this workload / batch."""
    try:
        with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles", "roofline_traffic.json")) as f:
            rec = json.load(f).get(workload)
        if rec and rec.get("batch_per_gpu") == batch:
            return {"traffic": rec["dram_bytes_per_step"], "traffic_unit": "bytes per step (all tc launches)",
                    "traffic_source": rec["source"]}
    except Exception:  # noqa: BLE001
        pass
    return {"traffic": None}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", os.environ.get("FDX_BENCH_SMI_MS", "200"), "-i", str(self.gpu)],
                                         stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:  # noqa: BLE001
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
                for n, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:  # noqa: BLE001
                pass
        sm.sort()
        # median of the upper half ~ clocks under load (idle samples at the edges excluded)
        load = sm[len(sm) // 2:] if sm else []
        return {"sm_mhz": (load[len(load) // 2] if load else None), "sm_max_mhz": (max(mx) if mx else None),
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------ reference arm
def run_reference(args):
    """CPU reference arm: the oracle restatement of the reference's train step on the host cores."""
    import torch
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from flaxdiff_b200.models.simple_unet import Unet
    from oracle import train_ref
    res, _, acfg, desc = WORKLOADS[args.workload]
    cores = usable_cores()
    torch.set_num_threads(cores)
    B = args.ref_batch
    model = Unet(attention_configs=acfg)
    fp = model.init(4, device=torch.device("cpu"))
    P = {k: v.clone().requires_grad_(True) for k, v in fp.named.items()}
    ema = {k: v.detach().clone() for k, v in P.items()}
    freqs = model._fourier_freqs("cpu")
    g = torch.Generator().manual_seed(0)
    img = torch.randint(0, 256, (B, res, res, 3), dtype=torch.uint8, generator=g)
    opt = {}
    times = []
    steps = max(1, min(args.steps, args.ref_max_steps))
    warm = max(1, min(args.warmup, 1))
    for i in range(warm + steps):
        noise = torch.randn(B, res, res, 3, generator=g)
        t = torch.randn(B, generator=g)
        t0 = time.perf_counter()
        train_ref.edm_train_step(P, opt, img, noise, t, freqs, attention_configs=acfg, ema=ema, step=i + 1)
        dt = time.perf_counter() - t0
        if i >= warm:
            times.append(dt)
    ms = 1e3 * sum(times) / len(times)
    val = B / (ms / 1e3)
    # sampler evaluations on the CPU
    x = torch.randn(B, res, res, 3, generator=g) * 80
    t0 = time.perf_counter()
    train_ref.karras_denoise_eval(P, x, torch.full((B,), 0.5), freqs, attention_configs=acfg)
    ev = time.perf_counter() - t0
    out = {
        "impl": "reference", "metric": "train_images_per_sec", "value": val, "unit": "images/s",
        "n_gpus": args.gpus, "steps": steps, "warmup": warm, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": desc, "sample": f"CPU oracle train step on B={B} images per step ({steps} timed)",
                   "resolution": res, "ref_batch": B, "ref_steps": steps,
                   "note": "bounded sample of the workload: the oracle port (the JAX reference is not installable) "
                           "at a reduced batch and step count so the run ends within minutes"},
        "cpu_baseline": {"value": val, "unit": "images/s", "cores": cores, "cpu": cpu_model(), "kind": "port",
                         "sample": f"oracle/train_ref.edm_train_step, B={B}, {steps} steps, torch fp32, {cores} threads",
                         "sample_unet_evals_per_sec": B / ev},
        "e2e": {"value": val, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(out)


# ------------------------------------------------------------------------------------------ this repo
def log(msg):
    if os.environ.get("FDX_BENCH_VERBOSE"):
        sys.stderr.write(f"[bench {time.strftime('%H:%M:%S')}] {msg}\n")
        sys.stderr.flush()


def cpu_model() -> str:
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except Exception:  # noqa: BLE001
        pass
    return "unknown"


class Dist:
    """rank / world / device of this process (torchrun env), NCCL group for the timing plumbing."""

    def __init__(self):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        torch.cuda.set_device(self.local_rank)
        self.dev = torch.device("cuda", self.local_rank)
        if self.world > 1 and not dist.is_initialized():
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            dist.init_process_group("nccl", device_id=self.dev)

    def sync(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_ms(self, *vals):
        t = self.torch.tensor(list(vals), device=self.dev, dtype=self.torch.float64)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return [float(v) for v in t]

    def close(self):
        if self.world > 1:
            self.dist.destroy_process_group()


def kernel_traffic(workload: str, kernel: str):
    """Per-launch DRAM bytes (dram__bytes_read.sum + dram__bytes_write.sum) of `kernel` from the committed ncu
    pass of the same workload (profiles/roofline_traffic.json, written by profiles/summarize_metrics.py)."""
    try:
        with open(os.path.join(ROOT, "profiles", "roofline_traffic.json")) as f:
            kern = json.load(f).get(workload, {}).get("kernels", {})
        # the ncu names carry the template arguments ("fdx_tc_kernel<256, 1, 2, 0>"): all instantiations of the family
        recs = [v for k, v in kern.items() if k == kernel or k.startswith(kernel + "<")]
        n = sum(r["launches"] for r in recs)
        if n:
            return {"traffic": sum(r["dram_bytes_per_launch"] * r["launches"] for r in recs) / n,
                    "traffic_unit": "DRAM bytes per launch (ncu, mean over the family's launches in one step)",
                    "traffic_launches": n, "traffic_source": recs[0]["source"]}
    except Exception:  # noqa: BLE001
        pass
    return {"traffic": None}


def profile_kernels(trainer, images, noise, t, ctx=None):
    """CUDA-event time and algorithmic FLOPs of every tensor-core launch in one EAGER training step, grouped
    by the kernel that actually ran (libfdx reports the family of its last launch).  One stream, no side
    stream / micro-batching: a kernel's duration only means something when it runs alone."""
    import torch
    from flaxdiff_b200 import _lib, ops
    lib = _lib.load()
    lib.fdx_kernel_kind_name.restype = __import__("ctypes").c_char_p

    def conv_flops(n, h, w, cin, cout):
        return 2.0 * n * h * w * 9 * cin * cout

    def f_fwd(a, k):
        x, wgt = a[0], a[1]
        st = k.get("stride", 1)
        return conv_flops(x.shape[0], -(-x.shape[1] // st), -(-x.shape[2] // st), x.shape[3], wgt.shape[-1])

    def f_dgrad(a, k):
        dy, wgt = a[0], a[1]
        return conv_flops(dy.shape[0], dy.shape[1], dy.shape[2], wgt.shape[2], wgt.shape[3])

    def f_wgrad(a, k):
        x, dy = a[0], a[1]
        return conv_flops(dy.shape[0], dy.shape[1], dy.shape[2], x.shape[3], dy.shape[3])

    def f_gemm(a, k):
        M, N, K = a[4], a[5], a[6]
        return 2.0 * M * N * K * max(1, k.get("batch1", 1)) * max(1, k.get("batch2", 1))

    def f_up_fwd(a, k):      # the reference's FLOPs: a 3x3 conv at the OUTPUT resolution (common.py:210-226)
        x, out = a[0], a[3]
        return conv_flops(out.shape[0], out.shape[1], out.shape[2], x.shape[3], out.shape[3])

    def f_up_dgrad(a, k):
        dy, dx = a[0], a[2]
        return conv_flops(dy.shape[0], dy.shape[1], dy.shape[2], dx.shape[3], dy.shape[3])

    def f_attn_fwd(a, k):    # q, k, v, heads, dh, scale: QK^T + PV at the TRUE head width (1 / scale^2)
        q, kk, heads, scale = a[0], a[1], a[3], a[5]
        return 4.0 * q.shape[0] * heads * q.shape[1] * kk.shape[1] * round(scale ** -2)

    def f_attn_bwd(a, k):    # q, k, v, o, lse, d_o, heads, dh, scale: dV, dP, dQ, dK
        q, kk, heads, scale = a[0], a[1], a[6], a[8]
        return 8.0 * q.shape[0] * heads * q.shape[1] * kk.shape[1] * round(scale ** -2)

    def f_1x1(a, k):         # x / dy (NHWC), w [.., Cin, Cout]: 1x1 convolution in conv geometry (fwd and dgrad)
        x, wgt = a[0], a[1]
        return 2.0 * x.shape[0] * x.shape[1] * x.shape[2] * wgt.shape[-2] * wgt.shape[-1]

    table = {"conv3x3_fwd": f_fwd, "conv3x3_dgrad": f_dgrad, "conv3x3_dgrad_gn": f_dgrad, "conv3x3_wgrad": f_wgrad,
             "conv1x1_fwd": f_1x1, "conv1x1_dgrad": f_1x1, "gemm": f_gemm,
             "upconv3x3_fwd": f_up_fwd, "upconv3x3_dgrad": f_up_dgrad, "upconv3x3_wgrad": f_wgrad,
             "attention_fwd": f_attn_fwd, "attention_bwd": f_attn_bwd}
    orig = {n: getattr(ops, n) for n in table}
    recs = []

    def shape_of(name, a, k):
        if name == "gemm":
            return f"M={a[4]} N={a[5]} K={a[6]} mode={a[0]} batch={k.get('batch1', 1)}x{k.get('batch2', 1)}"
        ts = [tuple(x.shape) for x in a[:4] if hasattr(x, "shape") and x.dim() == 4]
        return " ".join("x".join(map(str, t)) for t in ts[:2]) + (f" s{k['stride']}" if k.get("stride", 1) != 1 else "")

    def wrap(name, fn):
        def inner(*a, **k):
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            r = fn(*a, **k)
            e.record()
            kind = lib.fdx_last_kernel_kind()
            recs.append((s, e, table[name](a, k), kind, name, shape_of(name, a, k)))
            return r
        return inner
    saved_env = {k: os.environ.get(k) for k in ("FDX_MICROBATCH", "FDX_NO_SIDE")}
    os.environ["FDX_MICROBATCH"] = "1"
    os.environ["FDX_NO_SIDE"] = "1"
    overlap = trainer._overlap
    trainer._overlap = False                 # no NCCL kernels between the timed launches
    try:
        for n in table:
            setattr(ops, n, wrap(n, orig[n]))
        args = (images, noise, t) if ctx is None else (images, noise, t, ctx)
        trainer._fwd_bwd(*args)
        torch.cuda.synchronize()
    finally:
        for n in table:
            setattr(ops, n, orig[n])
        trainer._overlap = overlap
        for k, v in saved_env.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
    kinds = {}
    dump = os.environ.get("FDX_BENCH_CALLS")          # per-call table (op, shape, kernel, ms, TFLOP/s) for profiles/
    rows = []
    for s, e, fl, kind, name, shp in recs:
        kname = lib.fdx_kernel_kind_name(kind).decode()
        if dump:
            ms = s.elapsed_time(e)
            rows.append(f"{name:16s} {shp:44s} {kname:20s} {ms * 1e3:9.1f} us {fl / 1e9:9.1f} GF "
                        f"{fl / max(ms, 1e-6) / 1e9:8.1f} TF/s")
        d = kinds.setdefault(kname, {"calls": 0, "ms": 0.0, "gflop": 0.0})
        d["calls"] += 1
        d["ms"] += s.elapsed_time(e)
        d["gflop"] += fl / 1e9
    if dump:
        with open(dump, "w") as f:
            f.write("\n".join(rows) + "\n")
    return kinds


def run_train(D, args, workload, steps, warmup, with_cpu_baseline):
    """Training throughput of one workload: device-resident `value`, end-to-end `e2e` (pinned-host uint8 batch
    copied in + loss read back every step), launches, per-kernel roofline."""
    import torch
    from flaxdiff_b200 import _lib
    from flaxdiff_b200.inputs import DiffusionInputConfig
    from flaxdiff_b200.models.simple_unet import Unet
    from flaxdiff_b200.predictors import KarrasPredictionTransform
    from flaxdiff_b200.schedulers import EDMNoiseScheduler
    from flaxdiff_b200.trainer import GeneralDiffusionTrainer, adamw
    lib = _lib.load()
    lib.fdx_launch_count.restype = __import__("ctypes").c_ulonglong
    dev, rank, world = D.dev, D.rank, D.world
    res, B, acfg, desc = WORKLOADS[workload]
    if args.batch:
        B = args.batch
    model = Unet(attention_configs=acfg, dtype=torch.bfloat16)
    trainer = GeneralDiffusionTrainer(
        model, adamw(2.7e-4), EDMNoiseScheduler(1, sigma_max=80, rho=7, sigma_data=0.5),
        DiffusionInputConfig("image", (res, res, 3), []), rngs=4, name="bench",
        model_output_transform=KarrasPredictionTransform(sigma_data=0.5), ema_decay=0.999, device=dev,
        use_cuda_graph=not args.no_graph)
    step_fn = trainer._define_train_step(B)
    gen = torch.Generator().manual_seed(1234 + rank)
    host_batches = [torch.randint(0, 256, (B, res, res, 3), dtype=torch.uint8, generator=gen).pin_memory()
                    for _ in range(2)]
    dev_batch = host_batches[0].to(dev)
    E = res * res * 3
    fwd_gflop = FWD_GFLOP[(workload, res)]
    log(f'{workload}: trainer built')
    for i in range(warmup):
        trainer.state, loss, trainer.rngstate = step_fn(trainer.state, trainer.rngstate, {"image": dev_batch}, rank)
        torch.cuda.synchronize()
    clocks = ClockSampler(D.local_rank)
    D.sync()
    clocks.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        trainer.state, loss, trainer.rngstate = step_fn(trainer.state, trainer.rngstate, {"image": dev_batch}, rank)
    e1.record()
    D.sync()
    ms_dev = e0.elapsed_time(e1) / steps
    for i in range(2):                                  # untimed: first touch of each pinned batch / .item() path
        trainer.state, loss, trainer.rngstate = step_fn(trainer.state, trainer.rngstate,
                                                        {"image": host_batches[i % 2]}, rank)
        float(loss.item())
    D.sync()
    e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e2.record()
    last = 0.0
    for i in range(steps):
        trainer.state, loss, trainer.rngstate = step_fn(trainer.state, trainer.rngstate,
                                                        {"image": host_batches[i % 2]}, rank)
        last = float(loss.item())                       # device -> host read of the step's result
    e3.record()
    D.sync()
    clk = clocks.stop()
    st = trainer.state
    for name, t in (("loss", loss), ("params", st.params.flat), ("ema_params", st.ema_params.flat),
                    ("adam_mu", st.opt_state["mu"]), ("adam_nu", st.opt_state["nu"])):
        keep_output(f"{workload}_train_{name}", t)
    ms_e2e = e2.elapsed_time(e3) / steps
    ms_dev, ms_e2e = D.max_ms(ms_dev, ms_e2e)
    log(f'{workload}: {ms_dev:.2f} ms/step device, {ms_e2e:.2f} e2e')
    # launches per step: one eager (graph-less) fwd/bwd, counted by libfdx
    l1 = lib.fdx_launch_count()
    noise = torch.randn(B, res, res, 3, device=dev)
    tt = torch.randn(B, device=dev)
    trainer._fwd_bwd(dev_batch, noise, tt)
    torch.cuda.synchronize()
    launches_per_step = int(lib.fdx_launch_count() - l1) + 1   # + the fused optimiser kernel
    kinds = profile_kernels(trainer, dev_batch, noise, tt)
    hbm, tf_burst, tf_sust, src = load_peaks()
    step_tflop = 3 * fwd_gflop * B / 1e3
    out = None
    if rank == 0:
        for k, d in kinds.items():
            d["tflops"] = d["gflop"] / d["ms"] if d["ms"] > 0 else 0.0
            d["frac"] = d["tflops"] / tf_sust
            d["share_of_step"] = d["ms"] / ms_dev
        tc_ms = sum(d["ms"] for d in kinds.values())
        dom = max(kinds, key=lambda k: kinds[k]["ms"])
        dd = kinds[dom]
        out = {
            "value": world * B / (ms_dev / 1e3), "ms_per_step": ms_dev,
            "config": {"workload": desc, "resolution": res, "batch_per_gpu": B, "global_batch": B * world,
                       "parallelism": f"dp{world}", "params": model.layout().num_params,
                       "cuda_graph": not args.no_graph,
                       "grad_exchange": (f"fdx_comm_allreduce_avg x{len(trainer._exchange.bounds)} buckets, "
                                         "overlapped with backward" if trainer._overlap else
                                         "one fdx_comm_allreduce_avg (gradient + loss) after backward")
                       if trainer._exchange is not None else "none (single GPU)",
                       "l2": "per-step activation traffic (>= 9 GB) exceeds the 126 MB L2; no explicit flush needed"},
            "e2e": {"value": world * B / (ms_e2e / 1e3), "unit": "images/s", "ms_per_step": ms_e2e,
                    "h2d_bytes_per_step": B * E, "d2h_bytes_per_step": 4, "last_loss": last},
            "gpu_launches": launches_per_step * steps, "launches_per_step": launches_per_step,
            "train_tflops": step_tflop / (ms_dev / 1e3),
            "train_frac_of_sustained_bf16": step_tflop / (ms_dev / 1e3) / tf_sust,
            "roofline": {"bound": "tensor", "kernel": dom,
                         "why": "the tensor-core kernel with the largest share of the step (CUDA events around "
                                "each of its launches in one eager step; FLOPs = the reference's per layer)",
                         "achieved": dd["tflops"], "peak": tf_sust, "unit": "TFLOP/s", "frac": dd["frac"],
                         "peak_source": f"{src} bf16_tflops_sustained", "launches": dd["calls"],
                         "avg_launch_us": 1e3 * dd["ms"] / dd["calls"], "ms_in_step": dd["ms"],
                         "share_of_step": dd["share_of_step"], **kernel_traffic(workload, dom),
                         "all_tensor_kernels": {"ms_in_step": tc_ms, "share_of_step": tc_ms / ms_dev,
                                                "tflops": step_tflop / (tc_ms / 1e3),
                                                "frac": step_tflop / (tc_ms / 1e3) / tf_sust},
                         "kernels": kinds},
            "clocks": clk,
        }
        if with_cpu_baseline and not args.no_cpu_baseline:
            out["cpu_baseline"] = cpu_baseline(args, model, res, acfg)
    return out, trainer, model


def run_euler_c2(D, args, trainer, model, workload="c2"):
    import torch
    from flaxdiff_b200.inputs import DiffusionInputConfig
    from flaxdiff_b200.predictors import KarrasPredictionTransform
    from flaxdiff_b200.samplers import EulerSampler
    from flaxdiff_b200.schedulers import KarrasVENoiseScheduler
    res, B, acfg, desc = WORKLOADS[workload]
    if args.batch:
        B = args.batch
    dev, world = D.dev, D.world
    hbm, tf_burst, tf_sust, src = load_peaks()
    fwd_gflop = FWD_GFLOP[(workload, res)]
    sampler = EulerSampler(model, KarrasVENoiseScheduler(1, sigma_max=80, rho=7, sigma_data=0.5).to(dev),
                           KarrasPredictionTransform(0.5), DiffusionInputConfig("image", (res, res, 3), []))
    params = trainer.state.ema_params
    n_s = args.sample_steps
    sampler.generate_samples(params, B, res, diffusion_steps=min(n_s, 4), start_step=1000, device=dev)  # warm + capture
    D.sync()
    s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s0.record()
    imgs = sampler.generate_samples(params, B, res, diffusion_steps=n_s, start_step=1000, device=dev)
    s1.record()
    D.sync()
    keep_output(f"{workload}_sample{n_s}_images", imgs)
    (ms_s,) = D.max_ms(s0.elapsed_time(s1))
    return {"sampler": "EulerSampler", "diffusion_steps": n_s, "batch_per_gpu": B,
            "denoise_steps_per_sec": n_s / (ms_s / 1e3), "image_steps_per_sec": world * B * n_s / (ms_s / 1e3),
            "ms_per_denoise_step": ms_s / n_s,
            "tensor_frac_of_sustained": (fwd_gflop * B * n_s / 1e3) / (ms_s / 1e3) / tf_sust,
            "finite": bool(torch.isfinite(imgs).all().item())}


def sampling_runs(D, args, workload):
    """c4 (CFG Euler-ancestral, text cross-attention) / c5 (Heun sweep): replicas, no collective."""
    import torch
    from flaxdiff_b200.inputs import ConditionalInputConfig, DiffusionInputConfig, RandomEmbeddingEncoder
    from flaxdiff_b200.models.simple_unet import Unet
    from flaxdiff_b200.predictors import KarrasPredictionTransform
    from flaxdiff_b200.samplers import EulerAncestralSampler, HeunSampler
    from flaxdiff_b200.schedulers import KarrasVENoiseScheduler
    dev, rank, world = D.dev, D.rank, D.world
    res, B, acfg, desc = WORKLOADS[workload]
    if args.batch:
        B = args.batch
    hbm, tf_burst, tf_sust, src = load_peaks()
    sched = KarrasVENoiseScheduler(1, sigma_max=80, rho=7, sigma_data=0.5).to(dev)
    tr = KarrasPredictionTransform(0.5)
    fwd = FWD_GFLOP[(workload, res)]
    runs = []
    if workload == "c4":
        enc = RandomEmbeddingEncoder(77, 768, device=dev)
        cfg = DiffusionInputConfig("image", (res, res, 3), [ConditionalInputConfig(enc)])
        model = Unet(attention_configs=acfg, dtype=torch.bfloat16, context_dim=768)
        params = model.init(4 + rank, device=dev)
        smp = EulerAncestralSampler(model, sched, tr, cfg, guidance_scale=3.0)
        cond = (enc([f"prompt {i}" for i in range(B)]).to(dev),)
        plan = [(smp, 30, 2 * 30)]            # CFG doubles the model batch: 2 UNet evals per image-step
    else:
        cfg = DiffusionInputConfig("image", (res, res, 3), [])
        model = Unet(attention_configs=acfg, dtype=torch.bfloat16)
        params = model.init(4 + rank, device=dev)
        smp = HeunSampler(model, sched, tr, cfg)
        cond = ()
        plan = [(smp, n, 2 * n - 1) for n in (18, 50, 100)]
    clocks = ClockSampler(D.local_rank)
    first = True
    for smp_, n, nfe in plan:
        smp_.generate_samples(params, B, res, diffusion_steps=min(n, 3), start_step=1000, device=dev,
                              model_conditioning_inputs=cond)          # warm-up + graph capture
        D.sync()
        if first:
            clocks.start()
            first = False
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record()
        img = smp_.generate_samples(params, B, res, diffusion_steps=n, start_step=1000, device=dev,
                                    model_conditioning_inputs=cond)
        s1.record()
        D.sync()
        keep_output(f"{workload}_sample{n}_images", img)
        (ms,) = D.max_ms(s0.elapsed_time(s1))
        runs.append({"diffusion_steps": n, "unet_evals_per_image": nfe, "ms": ms,
                     "denoise_steps_per_sec": n / (ms / 1e3), "image_steps_per_sec": world * B * n / (ms / 1e3),
                     "unet_image_evals_per_sec": world * B * nfe / (ms / 1e3),
                     "tensor_frac_of_sustained": (fwd * B * nfe / 1e3) / (ms / 1e3) / tf_sust,
                     "finite": bool(torch.isfinite(img).all().item())})
    clk = clocks.stop()
    return {"workload": desc, "resolution": res, "batch_per_gpu": B, "parallelism": f"replicas{world}",
            "sampler": type(smp).__name__, "cuda_graph": True, "runs": runs, "clocks": clk}


def main():
    global _OUTPUTS
    claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="fdx", choices=["fdx", "reference"])
    ap.add_argument("--workload", default="all", choices=["all"] + sorted(WORKLOADS),
                    help="all (default) = the whole BASELINE metric: C2 train + Euler at 64x64, C3 train at 256x256, "
                         "C5 Heun sweep and C4 CFG sampling at 256x256; or one workload alone")
    ap.add_argument("--batch", type=int, default=0, help="override per-GPU batch (single-workload runs)")
    ap.add_argument("--sample-steps", type=int, default=50)
    ap.add_argument("--no-sample", action="store_true")
    ap.add_argument("--no-256", action="store_true", help="skip the 256x256 blocks of the default run")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--ref-batch", type=int, default=16)
    ap.add_argument("--ref-max-steps", type=int, default=3)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the timed path computed in its last step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "fdx":
        ap.error("--dump-outputs records the fdx path only")
    import faulthandler
    faulthandler.enable()
    if os.environ.get("FDX_BENCH_WATCHDOG"):
        faulthandler.dump_traceback_later(int(os.environ["FDX_BENCH_WATCHDOG"]), repeat=True, file=sys.stderr)
    if args.impl == "reference":
        if args.workload == "all":
            args.workload = "c2"
        return run_reference(args)
    args.warmup = max(args.warmup, 3)
    import gc

    import torch
    D = Dist()
    hbm, tf_burst, tf_sust, src = load_peaks()
    if args.dump_outputs and D.rank == 0:
        _OUTPUTS = {}

    if args.workload in ("c4", "c5"):
        blk = sampling_runs(D, args, args.workload)
        if D.rank == 0:
            runs = blk["runs"]
            head = runs[0] if args.workload == "c4" else runs[1]
            emit({"metric": "denoise_steps_per_sec", "value": head["denoise_steps_per_sec"], "unit": "steps/s",
                  "n_gpus": D.world, "steps": head["diffusion_steps"], "warmup": 3,
                  "ms_per_step": head["ms"] / head["diffusion_steps"], "higher_is_better": True, "scaling": "weak",
                  "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
                  "config": {k: blk[k] for k in ("workload", "resolution", "batch_per_gpu", "parallelism", "sampler",
                                                 "cuda_graph")},
                  "runs": runs, "clocks": blk["clocks"],
                  "roofline": {"bound": "tensor", "kernel": "UNet denoise evaluation (all libfdx launches of one step)",
                               "achieved": head["tensor_frac_of_sustained"] * tf_sust, "peak": tf_sust,
                               "unit": "TFLOP/s", "frac": head["tensor_frac_of_sustained"],
                               "peak_source": f"{src} bf16_tflops_sustained", "traffic": None}})
            if _OUTPUTS is not None:
                write_outputs(args.dump_outputs)
        return D.close()

    first = "c2" if args.workload == "all" else args.workload
    blk, trainer, model = run_train(D, args, first, args.steps, args.warmup, with_cpu_baseline=True)
    sample = None
    if not args.no_sample and first == "c2":
        sample = run_euler_c2(D, args, trainer, model)
    del trainer, model
    gc.collect()
    torch.cuda.empty_cache()
    extra = {}
    if args.workload == "all" and not args.no_256:
        # the 256x256 half of the metric: C3 training (B = 64 per GPU: global 512 at --gpus 8 = BASELINE
        # configs[2]), C5 Heun sweep and C4 CFG sampling as per-GPU replicas
        b3, tr3, m3 = run_train(D, args, "c3", args.steps, 3, with_cpu_baseline=False)
        del tr3, m3
        gc.collect()
        torch.cuda.empty_cache()
        if b3 is not None:
            b3.update({"metric": "train_images_per_sec", "unit": "images/s", "steps": args.steps, "warmup": 3})
        extra["train_256"] = b3
        if not args.no_sample:
            extra["sample_256_heun"] = sampling_runs(D, args, "c5")
            gc.collect()
            torch.cuda.empty_cache()
            extra["sample_256_text_cfg"] = sampling_runs(D, args, "c4")
    if D.rank == 0:
        out = {"metric": "train_images_per_sec", "value": blk["value"], "unit": "images/s", "n_gpus": D.world,
               "steps": args.steps, "warmup": args.warmup, "ms_per_step": blk["ms_per_step"],
               "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
               "data": "synthetic"}
        out.update({k: v for k, v in blk.items() if k not in ("value", "ms_per_step")})
        out["sample"] = sample
        out.update(extra)
        emit(out)
        if _OUTPUTS is not None:
            write_outputs(args.dump_outputs)
    D.close()


def cpu_baseline(args, model, res, acfg):
    """The oracle train step timed on the host cores on a bounded sample (rank 0, N=1 only)."""
    import torch
    from oracle import train_ref
    cores = usable_cores()
    torch.set_num_threads(cores)
    B = args.ref_batch
    fp = model.init(4, device=torch.device("cpu"))
    P = {k: v.clone().requires_grad_(True) for k, v in fp.named.items()}
    freqs = model._fourier_freqs("cpu")
    g = torch.Generator().manual_seed(0)
    img = torch.randint(0, 256, (B, res, res, 3), dtype=torch.uint8, generator=g)
    opt = {}
    times = []
    n = 2 if res <= 64 else 1
    for i in range(1 + n):
        noise = torch.randn(B, res, res, 3, generator=g)
        t = torch.randn(B, generator=g)
        t0 = time.perf_counter()
        train_ref.edm_train_step(P, opt, img, noise, t, freqs, attention_configs=acfg, step=i + 1)
        if i >= 1:
            times.append(time.perf_counter() - t0)
    sec = sum(times) / len(times)
    return {"value": B / sec, "unit": "images/s", "cores": cores, "cpu": cpu_model(), "kind": "port",
            "sample": f"oracle/train_ref.edm_train_step on B={B} images at {res}x{res}, {n} timed step(s), torch fp32"}


if __name__ == "__main__":
    main()
