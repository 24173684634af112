"""Training: `TrainState`, optimiser descriptions, `DynamicScale` and `GeneralDiffusionTrainer`
(API of flaxdiff/trainer/{diffusion_trainer.py:27-37, general_diffusion_trainer.py:108-518,
simple_trainer.py:341-389,500-677}).

One training step (general_diffusion_trainer.py:248-336) is, on each GPU:
    normalise + noise-add + precondition      fdx_diffuse_forward          (1 kernel)
    UNet forward / loss / UNet backward       Unet.forward / fdx_loss_fwd_bwd / Unet.backward
    gradient + loss mean over ranks           fdx_comm_allreduce_avg on BUCKETS of the flat f32 gradient
                                              buffer, each launched on a side stream as soon as the backward
                                              pass has finished the parameters it covers (the loss scalar
                                              rides in the tail of the first bucket launched)
    [clip / DynamicScale statistics]          fdx_grad_stats
    optimiser + EMA + bf16 shadow refresh     fdx_optimizer_step           (1 kernel; lamb: 2)
The forward/backward part - including the bucketed NCCL calls - is captured in a CUDA graph after the
first (eager) step; timesteps and noise are drawn outside the graph.  Out of scope (SURVEY.md $2.1 row 4):
wandb, registry pushes, AutoEncoderTrainer.
"""
from __future__ import annotations

import math
import os
import queue
import threading
import time
from dataclasses import dataclass, replace
from typing import Any, Callable, Dict, List, Optional, Tuple, Type, Union

import numpy as np
import torch

from .. import checkpoint as ckpt_io
from .. import ops, utils
from .._lib import OPT_ADAM, OPT_LAMB, FdxError
from ..models.params import FlatParams, from_tree
from ..predictors import DiffusionPredictionTransform, EpsilonPredictionTransform, _vec
from ..samplers import DDIMSampler, DiffusionSampler
from ..schedulers import NoiseScheduler
from ..utils import RandomMarkovState


# --------------------------------------------------------------------------- optimisers
@dataclass
class Optimizer:
    """Description of an optax chain (training.py:594-608): [clip_by_global_norm] -> adam / adamw / lamb."""
    learning_rate: Union[float, Callable[[int], float]] = 2.7e-4
    b1: float = 0.9
    b2: float = 0.999
    eps: float = 1e-8
    weight_decay: float = 0.0
    clip_norm: float = 0.0
    kind: str = "adamw"          # "adam" | "adamw" | "lamb"

    def lr_at(self, count: int) -> float:
        lr = self.learning_rate
        return float(lr(count)) if callable(lr) else float(lr)


def adam(learning_rate, b1=0.9, b2=0.999, eps=1e-8) -> Optimizer:
    return Optimizer(learning_rate, b1, b2, eps, 0.0, kind="adam")


def adamw(learning_rate, b1=0.9, b2=0.999, eps=1e-8, weight_decay=1e-4) -> Optimizer:
    return Optimizer(learning_rate, b1, b2, eps, weight_decay, kind="adamw")


def lamb(learning_rate, b1=0.9, b2=0.999, eps=1e-6, eps_root=0.0, weight_decay=0.0) -> Optimizer:
    """optax.lamb = scale_by_adam -> add_decayed_weights -> scale_by_trust_ratio -> -lr (training.py:266)."""
    if eps_root != 0.0:
        raise FdxError("lamb: eps_root != 0 is not supported")
    return Optimizer(learning_rate, b1, b2, eps, weight_decay, kind="lamb")


def clip_by_global_norm(max_norm: float) -> Optimizer:
    return Optimizer(clip_norm=max_norm, kind="clip")


def chain(*parts: Optimizer) -> Optimizer:
    out = Optimizer()
    for p in parts:
        if p.kind == "clip":
            out = replace(out, clip_norm=p.clip_norm)
        else:
            out = replace(p, clip_norm=out.clip_norm)
    return out


def warmup_cosine_decay_schedule(init_value, peak_value, warmup_steps, decay_steps, end_value=0.0):
    """optax.warmup_cosine_decay_schedule (training.py:263-267)."""
    def sched(count: int) -> float:
        if count < warmup_steps:
            return init_value + (peak_value - init_value) * count / max(warmup_steps, 1)
        t = min(max(count - warmup_steps, 0) / max(decay_steps - warmup_steps, 1), 1.0)
        return end_value + (peak_value - end_value) * 0.5 * (1 + math.cos(math.pi * t))
    return sched


class DynamicScale:
    """flax.training.dynamic_scale.DynamicScale (general_diffusion_trainer.py:305-318): the loss is multiplied
    by `scale` before the backward pass, the gradients are divided by it, a step with non-finite gradients
    leaves params / opt_state untouched and halves the scale; `growth_interval` finite steps in a row double
    it.  State lives on the device ({scale, fin_steps, last_is_finite}, f32[3]) so a CUDA-graph replay and the
    fused optimiser kernel read it without a host round trip."""

    def __init__(self, growth_factor: float = 2.0, backoff_factor: float = 0.5, growth_interval: int = 2000,
                 fin_steps: int = 0, scale: float = 65536.0, minimum_scale: float = float(np.finfo(np.float32).tiny)):
        self.growth_factor, self.backoff_factor = growth_factor, backoff_factor
        self.growth_interval, self.minimum_scale = growth_interval, minimum_scale
        self._init = (float(scale), float(fin_steps), 1.0)
        self.state: Optional[torch.Tensor] = None

    def to(self, device):
        if self.state is None or self.state.device != torch.device(device):
            self.state = torch.tensor(self._init, dtype=torch.float32, device=device)
        return self

    @property
    def scale(self) -> float:
        return float(self.state[0]) if self.state is not None else self._init[0]

    @property
    def fin_steps(self) -> int:
        return int(self.state[1]) if self.state is not None else int(self._init[1])

    def update(self, gstats: torch.Tensor):
        ops.dynscale_update(self.state, gstats, self.growth_factor, self.backoff_factor, self.growth_interval,
                            self.minimum_scale)


# --------------------------------------------------------------------------- data parallel
def dp_allreduce_sum_(grads_flat: torch.Tensor, loss: torch.Tensor, world_size: int) -> float:
    """The exchange step through `torch.distributed` (used for CPU / gloo process groups - the host-logic
    tests - and as the fallback when libfdx's NCCL binding is unavailable): sum all-reduce of the flat
    gradient buffer and of the scalar loss; returns the 1/world factor that turns the sums into the means
    (jax.lax.pmean, general_diffusion_trainer.py:325,334)."""
    if world_size <= 1:
        return 1.0
    torch.distributed.all_reduce(grads_flat)
    torch.distributed.all_reduce(loss)
    return 1.0 / world_size


def rank_key(key, rank: int):
    """Per-rank RNG stream: fold the rank into the step key (general_diffusion_trainer.py:251-253)."""
    return utils.fold_in(key, int(rank))


def bucket_bounds(total: int, n_buckets: int, align: int = 1024) -> List[Tuple[int, int]]:
    """[lo, hi) ranges covering [0, total), ascending, boundaries multiples of `align`."""
    n_buckets = max(1, int(n_buckets))
    edges = [0]
    for i in range(1, n_buckets):
        e = (total * i // n_buckets) // align * align
        if e > edges[-1]:
            edges.append(e)
    edges.append(total)
    return [(edges[i], edges[i + 1]) for i in range(len(edges) - 1)]


class GradExchange:
    """Bucketed, overlapped gradient mean (fdx_comm_allreduce_avg).  The backward pass finishes parameters
    from the END of the flat layout towards its start (the layout follows the forward order), so after the
    backward of a block whose first parameter sits at offset `lo` every bucket inside [lo, end) is final:
    `ready(lo, streams)` launches those buckets on the exchange stream behind events recorded on the
    producing streams; `finish()` launches what is left and joins.  The buffer's tail (64 floats after the
    parameters) carries the loss scalar, so it is averaged by the first bucket launched."""

    def __init__(self, comm: "ops.Comm", gbuf: torch.Tensor, n_buckets: int):
        self.comm, self.gbuf = comm, gbuf
        self.bounds = bucket_bounds(gbuf.numel(), n_buckets)
        self.stream = torch.cuda.Stream()
        self._next = len(self.bounds) - 1

    def begin(self):
        self._next = len(self.bounds) - 1

    def _launch_from(self, lo: int, streams):
        if self._next < 0 or self.bounds[self._next][0] < lo:
            return
        for s in streams:
            if s is not None:
                ev = torch.cuda.Event()
                ev.record(s)
                self.stream.wait_event(ev)
        while self._next >= 0 and self.bounds[self._next][0] >= lo:
            a, b = self.bounds[self._next]
            self.comm.allreduce_avg_(self.gbuf[a:b], self.stream)
            self._next -= 1

    def ready(self, lo: int, streams):
        self._launch_from(lo, streams)

    def finish(self, streams):
        self._launch_from(0, streams)
        torch.cuda.current_stream().wait_stream(self.stream)


_COMM: Optional["ops.Comm"] = None


def get_comm() -> Optional["ops.Comm"]:
    """Process-wide fdx_comm over the ranks of the default torch.distributed group (which is only used to
    hand the 128-byte NCCL id from rank 0 to the others).  None when not distributed / not NCCL."""
    global _COMM
    dist = torch.distributed
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() <= 1:
        return None
    if _COMM is not None:
        return _COMM
    if dist.get_backend() != "nccl" or os.environ.get("FDX_NO_COMM"):
        return None
    rank, world = dist.get_rank(), dist.get_world_size()
    box = [ops.Comm.unique_id() if rank == 0 else None]
    dist.broadcast_object_list(box, src=0)
    _COMM = ops.Comm(rank, world, box[0])
    return _COMM


# --------------------------------------------------------------------------- state
@dataclass
class TrainState:
    """flax TrainState + ema_params (trainer/diffusion_trainer.py:27-37).  Parameters, EMA and the Adam
    moments are flat f32 buffers with the model's layout; `apply_gradients` / `apply_ema` mutate them in
    place and return the state (the reference returns a new immutable pytree; callers that write
    `state = state.apply_gradients(grads=g).apply_ema(d)` behave identically)."""
    step: int
    params: FlatParams
    ema_params: FlatParams
    opt_state: Dict[str, Any]          # {'mu': flat f32, 'nu': flat f32, 'count': int}
    tx: Optimizer
    apply_fn: Callable = None
    rngs: Tuple[int, int] = (0, 0)
    dynamic_scale: Optional[DynamicScale] = None
    metrics: Any = None

    @classmethod
    def create(cls, apply_fn, params: FlatParams, ema_params: FlatParams, tx: Optimizer, rngs=(0, 0),
               dynamic_scale=None, metrics=None, **_):
        z = torch.zeros_like(params.flat)
        if dynamic_scale is not None:
            dynamic_scale.to(params.flat.device)
        return cls(0, params, ema_params, {"mu": z, "nu": z.clone(), "count": 0}, tx, apply_fn, tuple(rngs),
                   dynamic_scale, metrics)

    def replace(self, **kw) -> "TrainState":
        return replace(self, **kw)

    def clone(self) -> "TrainState":
        """Independent copy of every buffer (the reference's `best_state` is a separate pytree)."""
        return replace(self, params=self.params.clone(), ema_params=self.ema_params.clone(),
                       opt_state={"mu": self.opt_state["mu"].clone(), "nu": self.opt_state["nu"].clone(),
                                  "count": self.opt_state["count"]})

    # ---- the optimiser step ---------------------------------------------------------------------
    def _lamb_ws(self):
        ws = self.opt_state.get("_lamb")
        if ws is None:
            dev = self.params.flat.device
            offs = torch.tensor([o for o, _ in self.params.layout.table.values()], dtype=torch.int64, device=dev)
            ws = (offs, torch.empty(2 * offs.numel(), dtype=torch.float32, device=dev),
                  torch.empty_like(self.params.flat))
            self.opt_state["_lamb"] = ws
        return ws

    def _settle_count(self):
        """DynamicScale: a step whose gradients were not finite must not advance the optimiser count
        (general_diffusion_trainer.py:313-318 restores opt_state).  The flag of the PREVIOUS step is read
        here, lazily - one 4-byte read-back per step, only when loss scaling is on."""
        ds = self.dynamic_scale
        if ds is not None and self.opt_state.get("_ds_pending"):
            if float(ds.state[2]) == 0.0:
                self.opt_state["count"] -= 1
            self.opt_state["_ds_pending"] = False

    def _step(self, grads: FlatParams, ema: Optional[torch.Tensor], ema_decay: float, grad_scale: float,
              dyn: Optional[torch.Tensor]):
        tx = self.tx
        self._settle_count()
        count = self.opt_state["count"] + 1
        ds = self.dynamic_scale
        gstats = ops.grad_stats(grads.flat) if (tx.clip_norm > 0 or ds is not None) else None
        lr = tx.lr_at(count - 1)
        if dyn is not None:
            host = torch.tensor([lr, 1 - tx.b1 ** count, 1 - tx.b2 ** count], dtype=torch.float32)
            dyn.copy_(host, non_blocking=True)
        seg = (None, None, None)
        if tx.kind == "lamb":
            seg = self._lamb_ws()
        ops.optimizer_step(OPT_LAMB if tx.kind == "lamb" else OPT_ADAM, self.params.flat, grads.flat,
                           self.opt_state["mu"], self.opt_state["nu"], ema, self.params.shadow_flat_noupdate(),
                           lr, tx.b1, tx.b2, tx.eps, tx.weight_decay, count, ema_decay, grad_scale, gstats,
                           tx.clip_norm, dyn, ds.state if ds is not None else None, *seg)
        self.params.mark_shadow_fresh()
        if ema is not None:
            self.ema_params.touch()
        if ds is not None:
            ds.update(gstats)
            self.opt_state["_ds_pending"] = True
        self.opt_state["count"] = count
        self.step += 1
        return self

    def apply_gradients(self, *, grads: FlatParams, grad_scale: float = 1.0, dyn: torch.Tensor = None,
                        **_) -> "TrainState":
        """flax `TrainState.apply_gradients(grads=...)`: tx.update -> apply_updates -> step + 1
        (general_diffusion_trainer.py:311,327).  `grads` is a FlatParams or a flax-named tree."""
        if not isinstance(grads, FlatParams):
            grads = from_tree(self.params.layout, grads, self.params.flat.device)
        return self._step(grads, None, 0.0, grad_scale, dyn)

    def apply_ema(self, decay: float = 0.999) -> "TrainState":
        """ema = decay * ema + (1 - decay) * params (trainer/diffusion_trainer.py:31-37)."""
        ops.ema_update(self.ema_params.flat, self.params.flat, decay)
        self.ema_params.touch()
        return self

    def apply_gradients_and_ema(self, grads: FlatParams, ema_decay: float, grad_scale: float = 1.0,
                                dyn: torch.Tensor = None) -> "TrainState":
        """apply_gradients followed by apply_ema (general_diffusion_trainer.py:327-330) in ONE kernel."""
        return self._step(grads, self.ema_params.flat, ema_decay, grad_scale, dyn)


# --------------------------------------------------------------------------- host -> device prefetch
class DevicePrefetcher:
    """uint8 host -> device prefetch (the reference's daemon prefetch thread, data/dataloaders.py:28-82, plus
    jax.device_put): a background thread pulls batches from the iterator, stages the sample tensor in one of a
    small RING of pinned buffers (allocated once, in the constructor's thread: no cudaHostAlloc ever runs
    concurrently with a CUDA-graph capture) and copies it to the device on a copy stream, `depth` batches ahead
    of the consumer.  Yields batches whose sample entry is a device tensor usable on the current stream."""

    def __init__(self, it, key: str, device, depth: int = 2):
        self.it, self.key = iter(it), key
        dev = torch.device(device)
        if dev.type == "cuda" and dev.index is None:
            dev = torch.device("cuda", torch.cuda.current_device())
        self.device = dev
        self.depth = max(1, depth)
        self.q: "queue.Queue" = queue.Queue(maxsize=self.depth)
        self.stream = torch.cuda.Stream(device=self.device)
        self._stop = False
        self._ring: List[torch.Tensor] = []
        self._free: "queue.Queue" = queue.Queue()
        # the first batch is staged here, synchronously: it sizes the pinned ring
        try:
            first = next(self.it)
        except StopIteration:
            first = None
        if first is not None:
            data = self._as_tensor(first[self.key])
            for _ in range(self.depth + 2):
                buf = torch.empty(tuple(data.shape), dtype=data.dtype).pin_memory()
                self._ring.append(buf)
                self._free.put(buf)
            self.q.put(self._stage(first, data))
        self.th = threading.Thread(target=self._run, args=(first is None,), daemon=True)
        self.th.start()

    @staticmethod
    def _as_tensor(data):
        if not isinstance(data, torch.Tensor):
            data = torch.as_tensor(np.asarray(data))
        if data.dtype not in (torch.uint8, torch.float32):
            data = data.to(torch.float32)
        return data

    def _stage(self, batch, data):
        if self._ring and tuple(data.shape) == tuple(self._ring[0].shape) and data.dtype == self._ring[0].dtype:
            pinned = self._free.get()
            pinned.copy_(data)
        else:                                   # ragged last batch: one-off pinned copy
            pinned = data.contiguous().pin_memory()
        with torch.cuda.stream(self.stream):
            dev = pinned.to(self.device, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(self.stream)
        out = dict(batch)
        out[self.key] = dev
        return (out, ev, pinned)

    def _run(self, empty: bool):
        try:
            torch.cuda.set_device(self.device)
            if not empty:
                for batch in self.it:
                    if self._stop:
                        break
                    self.q.put(self._stage(batch, self._as_tensor(batch[self.key])))
            self.q.put(None)
        except BaseException as e:  # noqa: BLE001 - surfaced to the consumer
            self.q.put(e)

    def __iter__(self):
        return self

    def __next__(self):
        item = self.q.get()
        if item is None:
            raise StopIteration
        if isinstance(item, BaseException):
            raise item
        batch, ev, pinned = item
        torch.cuda.current_stream().wait_event(ev)
        batch[self.key].record_stream(torch.cuda.current_stream())
        if any(pinned is b for b in self._ring):
            ev.synchronize()                    # the H2D copy has left the pinned buffer: recycle it
            self._free.put(pinned)
        return batch

    def close(self):
        self._stop = True
        try:                                    # unblock a producer waiting on a full queue / an empty ring
            while True:
                self.q.get_nowait()
        except queue.Empty:
            pass
        for b in self._ring:
            self._free.put(b)


# --------------------------------------------------------------------------- trainer
class GeneralDiffusionTrainer:
    def __init__(self, model, optimizer: Optimizer, noise_schedule: NoiseScheduler, input_config,
                 rngs, unconditional_prob: float = 0.12, name: str = "GeneralDiffusion",
                 model_output_transform: DiffusionPredictionTransform = None, autoencoder=None,
                 native_resolution: int = None, frames_per_sample: int = None, wandb_config=None,
                 eval_metrics=None, best_tracker_metric: str = "train/best_loss",
                 distributed_training: bool = None, checkpoint_base_path: str = "./checkpoints",
                 use_dynamic_scale: bool = False, ema_decay: float = 0.999, device=None,
                 use_cuda_graph: bool = True, grad_buckets: int = None, **kwargs):
        if autoencoder is not None:
            raise FdxError("latent diffusion (autoencoder) is outside the supported hot path")
        self.model = model
        self.optimizer = optimizer
        self.noise_schedule = noise_schedule
        self.input_config = input_config
        self.model_output_transform = model_output_transform or EpsilonPredictionTransform()
        self.unconditional_prob = unconditional_prob
        self.name = name
        self.ema_decay = ema_decay
        self.autoencoder = None
        self.eval_metrics = eval_metrics
        self.best_val_metrics: Dict[str, float] = {}
        self.metric_higher_is_better: Dict[str, bool] = kwargs.get("metric_higher_is_better", {})
        self.checkpoint_base_path = checkpoint_base_path
        self.use_cuda_graph = use_cuda_graph
        self.use_dynamic_scale = use_dynamic_scale
        self.device = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        noise_schedule.to(self.device)
        shape = input_config.sample_data_shape
        self.native_resolution = native_resolution or shape[-2]
        dist = torch.distributed
        self.world_size = dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1
        self.rank = dist.get_rank() if self.world_size > 1 else 0
        self.distributed_training = (self.world_size > 1) if distributed_training is None else distributed_training
        if isinstance(rngs, int):
            rngs = utils.PRNGKey(rngs)
        self.rngstate = RandomMarkovState(tuple(rngs))
        self.state, self.best_state = self.generate_states(optimizer, tuple(rngs), model=model,
                                                           use_dynamic_scale=use_dynamic_scale)
        self.best_loss = 1e9
        self.latest_step = 0
        self._graph = None
        self._static = None
        self._dyn = torch.zeros(3, dtype=torch.float32, device=self.device)
        # gradient buffer = the parameter layout + a 64-float tail; tail[0] carries the loss through the
        # exchange (general_diffusion_trainer.py:334 pmean(loss))
        total = self.state.params.layout.total
        self._gbuf = torch.zeros(total + 64, dtype=torch.float32, device=self.device)
        self._grads = FlatParams(self.state.params.layout, self._gbuf[:total])
        self._comm = get_comm() if (self.distributed_training and self.device.type == "cuda") else None
        nb = grad_buckets if grad_buckets is not None else int(os.environ.get("FDX_GRAD_BUCKETS", "4"))
        self._exchange = GradExchange(self._comm, self._gbuf, nb) if self._comm is not None else None
        # one exchange after the backward unless FDX_NO_DP_OVERLAP is set to "0" (or ""): bucketed launches from the
        # backward inside the training graph measured slower on 8 B200s (DESIGN 5)
        self._overlap = self._exchange is not None and os.environ.get("FDX_NO_DP_OVERLAP") in ("", "0")

    # ------------------------------------------------------------------ state
    def generate_states(self, optimizer, rngs, existing_state=None, existing_best_state=None, model=None,
                        param_transforms=None, use_dynamic_scale=False):
        rngs, subkey = utils.split(rngs)
        model = model or self.model
        if existing_state is None:
            ctx_ex = None
            if self.input_config.conditions:
                ctx_ex = self.input_config.conditions[0].get_unconditional()
            params = model.init(subkey, textcontext=ctx_ex, device=self.device)
            ema = params.clone()
        else:
            params, ema = existing_state['params'], existing_state['ema_params']
            if not isinstance(params, FlatParams):
                params = from_tree(model.layout(), params, self.device)
            if not isinstance(ema, FlatParams):
                ema = from_tree(model.layout(), ema, self.device)
        if param_transforms is not None:
            params = param_transforms(params)
        ds = DynamicScale() if use_dynamic_scale else None
        state = TrainState.create(apply_fn=model.apply, params=params, ema_params=ema, tx=optimizer, rngs=rngs,
                                  dynamic_scale=ds)
        if existing_best_state is not None:
            bp, be = existing_best_state['params'], existing_best_state['ema_params']
            bp = bp if isinstance(bp, FlatParams) else from_tree(model.layout(), bp, self.device)
            be = be if isinstance(be, FlatParams) else from_tree(model.layout(), be, self.device)
            best = TrainState.create(apply_fn=model.apply, params=bp, ema_params=be, tx=optimizer, rngs=rngs)
        else:
            best = state.clone()             # an independent copy, as the reference's separate pytree
        return state, best

    # ------------------------------------------------------------------ the step
    def _fwd_bwd(self, images, noise, noise_level, ctx=None):
        """noise-add -> UNet fwd -> loss -> UNet bwd [-> bucketed gradient exchange]; returns the loss tensor
        (f32[1]); gradients land in self._grads.  FDX_MICROBATCH=2 processes the batch as two micro-batches
        on two streams; measured slower than one batch with side-stream weight gradients, hence opt-in."""
        B = images.shape[0]
        nmb = int(os.environ.get("FDX_MICROBATCH", "1"))
        if nmb < 2 or B % nmb != 0 or B // nmb < 2:
            return self._fwd_bwd_one(images, noise, noise_level, ctx, self._grads, exchange=True)
        if getattr(self, "_mb_grads", None) is None or len(self._mb_grads) != nmb:
            self._mb_grads = [self.state.params.zeros_like() for _ in range(nmb)]
            self._mb_streams = [torch.cuda.Stream() for _ in range(nmb)]
        main = torch.cuda.current_stream()
        ev = torch.cuda.Event()
        ev.record(main)
        losses = []
        step = B // nmb
        for h in range(nmb):
            sl = slice(h * step, (h + 1) * step)
            self._mb_streams[h].wait_event(ev)
            with torch.cuda.stream(self._mb_streams[h]):
                losses.append(self._fwd_bwd_one(images[sl], noise[sl], noise_level[sl],
                                                None if ctx is None else ctx[sl], self._mb_grads[h]))
        for h in range(nmb):
            main.wait_stream(self._mb_streams[h])
        g = self._grads.flat
        if nmb == 2:
            torch.lerp(self._mb_grads[0].flat, self._mb_grads[1].flat, 0.5, out=g)
        else:
            torch.add(self._mb_grads[0].flat, self._mb_grads[1].flat, out=g)
            for h in range(2, nmb):
                g.add_(self._mb_grads[h].flat)
            g.mul_(1.0 / nmb)
        loss = losses[0]
        for h in range(1, nmb):
            loss = loss + losses[h]
        loss = loss / nmb
        if self._overlap:
            self._gbuf[-64:-63].copy_(loss)
            self._exchange.begin()
            self._exchange.finish([torch.cuda.current_stream()])
            loss = self._gbuf[-64:-63]
        return loss

    def _fwd_bwd_one(self, images, noise, noise_level, ctx, grads, exchange=False):
        sched, tr, st = self.noise_schedule, self.model_output_transform, self.state
        B = images.shape[0]
        rates = sched.get_rates(noise_level, shape=(-1,))
        alpha, sigma = rates
        c_in = tr.get_input_scale(rates)
        c_in = _vec(c_in, B, images.device)
        c_out, c_skip = tr.loss_coeffs(rates)
        weight = sched.get_weights(noise_level, shape=(-1,)).to(torch.float32)
        _, t_model = sched.transform_inputs(None, noise_level)
        x_t, target, model_in = ops.diffuse_forward(images, noise, alpha, sigma, c_in, True, tr.target_kind)
        F, saved = self.model.forward(st.params, model_in, t_model, ctx, save=True)
        loss, dF = ops.loss_fwd_bwd(F, x_t, target, c_out, c_skip, weight, want_grad=True)
        ds = st.dynamic_scale
        if ds is not None:
            # DynamicScale.value_and_grad differentiates loss * scale (the optimiser divides it back out)
            dF, _, _ = ops.affine_combine([dF], ds.state[0:1].expand(1, B))
        grads.flat.zero_()
        overlap = exchange and self._overlap
        if overlap:
            self._gbuf[-64:-63].copy_(loss)
            self._exchange.begin()
            self.model.backward(st.params, saved, dF, grads, on_ready=self._exchange.ready)
            self._exchange.finish([torch.cuda.current_stream()])
            return self._gbuf[-64:-63]
        self.model.backward(st.params, saved, dF, grads)
        return loss

    def _define_train_step(self, batch_size=None):
        key = self.input_config.sample_data_key
        dev = self.device

        def train_step(train_state: TrainState, rng_state: RandomMarkovState, batch, local_device_index=None):
            rng_state, key_fold = rng_state.get_random_key()
            idx = self.rank if local_device_index is None else int(local_device_index)
            local = RandomMarkovState(rank_key(key_fold, idx))
            data = batch[key]
            if not isinstance(data, torch.Tensor):
                data = torch.as_tensor(data)
            if data.dtype not in (torch.uint8, torch.float32):
                data = data.to(torch.float32)
            images = data.to(dev, non_blocking=True).contiguous()      # HOST -> DEVICE boundary
            B = images.shape[0]
            local, uncond_key = local.get_random_key()
            ctx = None
            if self.input_config.conditions:
                # per-sample unconditional mask (bernoulli p = unconditional_prob) and null-embedding mixing
                # (general_diffusion_trainer.py:266-275; inputs/__init__.py:123-146)
                mask = utils.device_uniform(uncond_key, (B,), dev) < self.unconditional_prob
                ctx = self.input_config.process_conditioning(batch, uncond_mask=mask)[0]
                ctx = ctx.to(device=dev, dtype=torch.float32).contiguous()
            noise_level, local = self.noise_schedule.generate_timesteps(B, local)
            local, noise_key = local.get_random_key()
            noise = utils.device_normal(noise_key, tuple(images.shape), dev)
            if train_state is not self.state:
                self.state = train_state               # the step reads parameters through self.state
                self._graph = None
            if self.use_cuda_graph:
                loss = self._graphed_fwd_bwd(images, noise, noise_level, ctx)
            else:
                loss = self._fwd_bwd(images, noise, noise_level, ctx)
                if self._overlap:
                    loss = loss.clone()             # a view of the exchange buffer's tail otherwise
            gscale = 1.0
            if self.distributed_training and self.world_size > 1 and not self._overlap:
                if self._exchange is not None:           # one un-overlapped call over gradients + loss tail
                    self._gbuf[-64:-63].copy_(loss)
                    self._comm.allreduce_avg_(self._gbuf)
                    loss = self._gbuf[-64:-63].clone()
                else:                                    # torch.distributed (gloo on CPU tests)
                    gscale = dp_allreduce_sum_(self._grads.flat, loss, self.world_size)
                    loss = loss * gscale
            train_state.apply_gradients_and_ema(self._grads, self.ema_decay, gscale, self._dyn)
            return train_state, loss, rng_state

        return train_step

    def _graphed_fwd_bwd(self, images, noise, noise_level, ctx=None):
        if self._graph is None or self._static[0].shape != images.shape or self._static[0].dtype != images.dtype:
            self._static = [images.clone(), noise.clone(), noise_level.clone()]
            if ctx is not None:
                self._static.append(ctx.clone())
            self.state.params.shadow()              # bf16 weights current before warm-up and capture
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                self._fwd_bwd(*self._static)        # eager warm-up on a side stream
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            self._graph = torch.cuda.CUDAGraph()
            # other threads must stay free to call the CUDA API during the capture (NCCL's proxy thread for the
            # captured all-reduce launches, the DevicePrefetcher's pin_memory / copies) -> thread-local mode
            with torch.cuda.graph(self._graph, capture_error_mode="thread_local"):
                self._static_loss = self._fwd_bwd(*self._static)
        self._static[0].copy_(images, non_blocking=True)
        self._static[1].copy_(noise)
        self._static[2].copy_(noise_level)
        if ctx is not None:
            self._static[3].copy_(ctx)
        if not self.state.params.shadow_is_fresh():
            self.state.params.shadow()              # parameters changed outside the fused optimiser (load, ...)
        self._graph.replay()
        return self._static_loss.clone()

    # ------------------------------------------------------------------ validation / sampling
    def _get_image_size(self):
        if self.native_resolution is not None:
            return self.native_resolution
        return self.input_config.sample_data_shape[-2]

    def _define_validation_step(self, sampler_class: Type[DiffusionSampler] = DDIMSampler,
                                sampling_noise_schedule: NoiseScheduler = None):
        """general_diffusion_trainer.py:351-402: a sampler over the EMA weights with guidance 3.0."""
        sched = self.noise_schedule if sampling_noise_schedule is None else sampling_noise_schedule
        sched.to(self.device)
        sampler = sampler_class(model=self.model, noise_schedule=sched,
                                model_output_transform=self.model_output_transform, input_config=self.input_config,
                                autoencoder=None,
                                guidance_scale=3.0 if self.input_config.conditions else 0.0)
        image_size = self._get_image_size()
        conds = self.input_config.conditions

        def generate_samples(val_state: TrainState, batch, diffusion_steps: int):
            mci = [c(batch).to(self.device) for c in conds] if (conds and batch is not None) else []
            if conds and not mci:
                mci = [c.get_unconditional().to(self.device).expand(4, -1, -1).contiguous() for c in conds]
            batch_size = len(mci[0]) if mci else 4
            return sampler.generate_samples(params=val_state.ema_params, resolution=image_size,
                                            num_samples=batch_size, sequence_length=None,
                                            diffusion_steps=diffusion_steps, start_step=1000, end_step=0,
                                            priors=None, model_conditioning_inputs=tuple(mci), device=self.device)

        return generate_samples

    def validation_loop(self, val_state: TrainState, val_step_fn: Callable, val_ds, val_steps_per_epoch,
                        current_step, diffusion_steps=200):
        """general_diffusion_trainer.py:420-518 without wandb: draw samples from the EMA weights, evaluate
        the configured metrics; errors are caught and printed like the reference does."""
        val_it = iter(val_ds()) if val_ds else None
        samples = None
        try:
            metrics = {m.name: [] for m in self.eval_metrics} if self.eval_metrics else {}
            for _ in range(val_steps_per_epoch):
                batch = next(val_it) if val_it is not None else None
                samples = val_step_fn(val_state, batch, diffusion_steps)
                for m in (self.eval_metrics or []):
                    try:
                        metrics[m.name].append(float(m.function(samples, batch)))
                    except Exception as e:  # noqa: BLE001
                        print("Error in evaluation metrics:", e)
            for k, v in metrics.items():
                if not v:
                    continue
                val, fk = float(np.mean(v)), f"val/{k}"
                hib = self.metric_higher_is_better.get(fk, False)
                prev = self.best_val_metrics.get(fk)
                self.best_val_metrics[fk] = val if prev is None else (max(prev, val) if hib else min(prev, val))
        except StopIteration:
            print("Validation dataset exhausted")
        except FdxError:
            raise
        self.last_val_samples = samples
        return samples

    # ------------------------------------------------------------------ loops
    def train_loop(self, train_state, train_step_fn, train_ds, train_steps_per_epoch, current_step, rng_state,
                   verbose=False):
        epoch_loss = torch.zeros(1, dtype=torch.float32, device=self.device)
        for i in range(train_steps_per_epoch):
            batch = next(train_ds)
            train_state, loss, rng_state = train_step_fn(train_state, rng_state, batch, self.rank)
            epoch_loss += loss                      # accumulated on the device: no per-step host sync
            if i % 100 == 0:
                lv = float(loss.item())
                if not math.isfinite(lv) or lv <= 1e-8:
                    raise FdxError(f"loss became invalid ({lv}) at step {current_step + i}")
        return float(epoch_loss.item()), current_step + train_steps_per_epoch, train_state, rng_state

    def fit(self, data, training_steps_per_epoch=None, epochs=1, val_steps_per_epoch=8,
            sampler_class: Type[DiffusionSampler] = DDIMSampler, sampling_noise_schedule=None, verbose=True,
            train_steps_per_epoch=None, val_diffusion_steps: int = 200, save_checkpoints: bool = False,
            prefetch: int = 2):
        """Host loop of simple_trainer.py:601-677 / general_diffusion_trainer.py:520-: sanity validation,
        then per epoch train -> validation sampling from the EMA weights -> best-state tracking
        (-> orbax-layout checkpoint when `save_checkpoints`)."""
        steps_pe = training_steps_per_epoch if training_steps_per_epoch is not None else train_steps_per_epoch
        val_ds = data.get('val', data.get('test', None))
        step_fn = self._define_train_step(data.get('local_batch_size'))
        val_step = self._define_validation_step(sampler_class, sampling_noise_schedule)
        if val_steps_per_epoch > 0:
            # sanity validation first (it also captures the sampler's graphs before any background thread exists)
            self.validation_loop(self.state, val_step, val_ds, val_steps_per_epoch, self.latest_step,
                                 val_diffusion_steps)
        train_ds = iter(data['train']())
        if prefetch and self.device.type == "cuda":
            train_ds = DevicePrefetcher(train_ds, self.input_config.sample_data_key, self.device, prefetch)
        while self.latest_step < epochs * steps_pe:
            epoch = self.latest_step // steps_pe
            t0 = time.time()
            epoch_loss, cur, self.state, self.rngstate = self.train_loop(self.state, step_fn, train_ds, steps_pe,
                                                                         self.latest_step, self.rngstate)
            self.latest_step = cur
            dt = time.time() - t0
            if val_steps_per_epoch > 0:
                self.validation_loop(self.state, val_step, val_ds, val_steps_per_epoch, cur, val_diffusion_steps)
            avg = epoch_loss / steps_pe
            if avg < self.best_loss:
                self.best_loss = avg
                self.best_state = self.state.clone()
                if save_checkpoints:
                    self.save(epoch, cur)
            if verbose and self.rank == 0:
                print(f"epoch {epoch}: avg loss {avg:.5f}, {dt / steps_pe * 1e3:.1f} ms/step, best {self.best_loss:.5f}")
        if isinstance(train_ds, DevicePrefetcher):
            train_ds.close()
        if save_checkpoints:
            self.save(epochs, self.latest_step)
        return self.state

    def make_sampler(self, sampler_class: Type[DiffusionSampler] = DDIMSampler, sampling_noise_schedule=None,
                     guidance_scale: float = 0.0):
        return sampler_class(model=self.model, noise_schedule=sampling_noise_schedule or self.noise_schedule,
                             model_output_transform=self.model_output_transform, input_config=self.input_config,
                             guidance_scale=guidance_scale)

    # ------------------------------------------------------------------ checkpoints (orbax layout)
    def checkpoint_path(self) -> str:
        path = os.path.join(self.checkpoint_base_path, self.name.replace(' ', '_').lower())
        os.makedirs(path, exist_ok=True)
        return path

    @staticmethod
    def _state_tree(st: TrainState) -> dict:
        lay = st.params.layout
        mu = FlatParams(lay, st.opt_state["mu"])
        nu = FlatParams(lay, st.opt_state["nu"])
        out = {
            "step": np.asarray(st.step, dtype=np.int32),
            "params": _np_tree(st.params),
            "ema_params": _np_tree(st.ema_params),
            # optax adam / adamw / lamb state = (ScaleByAdamState(count, mu, nu), EmptyState())
            "opt_state": ({"count": np.asarray(st.opt_state["count"], dtype=np.int32),
                           "mu": _np_tree(mu), "nu": _np_tree(nu)}, None),
            "rngs": np.asarray(st.rngs, dtype=np.uint32),
        }
        if st.dynamic_scale is not None:
            ds = st.dynamic_scale
            out["dynamic_scale"] = {"fin_steps": np.asarray(ds.fin_steps, dtype=np.int32),
                                    "scale": np.asarray(ds.scale, dtype=np.float32)}
        return out

    def save(self, epoch=0, step=0, state=None, rngstate=None, path: str = None) -> str:
        """simple_trainer.py:371-389: {'rngs','state','best_state','best_loss','epoch'} in the orbax aggregate
        layout <checkpoint_path>/<step>/default/{checkpoint,_METADATA} (flaxdiff_b200/checkpoint.py)."""
        st = self.state if state is None else state
        rs = self.rngstate if rngstate is None else rngstate
        tree = {"rngs": {"rng": np.asarray(rs.rng, dtype=np.uint32)},
                "state": self._state_tree(st), "best_state": self._state_tree(self.best_state),
                "best_loss": np.asarray(self.best_loss, dtype=np.float64), "epoch": np.asarray(epoch)}
        return ckpt_io.save_tree(path or self.checkpoint_path(), step, tree)

    def _load_state_tree(self, st: TrainState, tree: dict):
        lay = st.params.layout
        names = list(lay.table)
        for key, fp in (("params", st.params), ("ema_params", st.ema_params)):
            got = sorted(ckpt_io.flatten_names(tree[key].get("params", tree[key])))
            if got != sorted(names):
                missing = [n for n in names if n not in got][:4]
                extra = [n for n in got if n not in lay.table][:4]
                raise FdxError(f"checkpoint {key} do not match this model: missing {missing}, unexpected {extra}")
            src = from_tree(lay, tree[key], fp.flat.device)
            fp.flat.copy_(src.flat)
            fp.touch()
        opt = tree["opt_state"]["0"] if "0" in tree["opt_state"] else tree["opt_state"][0]
        for key, buf in (("mu", st.opt_state["mu"]), ("nu", st.opt_state["nu"])):
            buf.copy_(from_tree(lay, opt[key], buf.device).flat)
        st.opt_state["count"] = int(np.asarray(opt["count"]))
        st.step = int(np.asarray(tree["step"]))
        if "rngs" in tree:
            st.rngs = tuple(int(x) for x in np.asarray(tree["rngs"]).reshape(-1)[:2])
        if st.dynamic_scale is not None and tree.get("dynamic_scale"):
            d = tree["dynamic_scale"]
            st.dynamic_scale.state.copy_(torch.tensor([float(np.asarray(d["scale"])),
                                                       float(np.asarray(d["fin_steps"])), 1.0]))
        # tensor-core kernels read the bf16 shadow; graphs captured for the old values stay valid (they read
        # the same buffers) but the shadow must follow the new f32 values
        st.params.shadow()
        st.ema_params.shadow()

    def load(self, checkpoint_path: str = None, checkpoint_step: int = None, load_directly_from_dir: bool = False):
        """simple_trainer.py:341-369: restores state / best_state / rngs / best_loss; returns
        (step, state, best_state, rngstate).  Raises when the tree does not match this model's layout."""
        base = checkpoint_path or self.checkpoint_path()
        step, ck = ckpt_io.load_tree(base, checkpoint_step, load_directly_from_dir)
        self._load_state_tree(self.state, ck["state"])
        if ck.get("best_state") is not None:
            self._load_state_tree(self.best_state, ck["best_state"])
        r = ck.get("rngs")
        if isinstance(r, dict):
            r = r.get("rng")
        if r is not None:
            self.rngstate = RandomMarkovState(tuple(int(x) for x in np.asarray(r).reshape(-1)[:2]))
        self.best_loss = float(np.asarray(ck["best_loss"]))
        if self.best_loss == 0:
            self.best_loss = 1e9
        self.latest_step = self.state.step
        return step, self.state, self.best_state, self.rngstate


def _np_tree(fp: FlatParams) -> dict:
    """{'params': nested numpy tree} view of a FlatParams (flax layouts: HWIO kernels, (in, out) dense)."""
    from ..models.params import nest
    return {"params": nest({k: v.detach().cpu().numpy() for k, v in fp.named.items()})}


DiffusionTrainer = GeneralDiffusionTrainer
SimpleTrainState = TrainState          # flaxdiff/trainer/simple_trainer.py:73-75 (same fields here: step, params,
                                       # opt state, dynamic scale; metrics live on the trainer)
from ..inputs import ConditionalInputConfig  # noqa: E402,F401  (re-exported by flaxdiff/trainer/__init__.py)


class Metrics:
    """Host-side stand-in for the clu metrics collection of flaxdiff/trainer/simple_trainer.py:68-70: a running
    average of the loss (`accuracy` is never filled by the diffusion trainers)."""

    def __init__(self, total: float = 0.0, count: int = 0):
        self.total, self.count = float(total), int(count)

    @classmethod
    def empty(cls) -> "Metrics":
        return cls()

    def single_from_model_output(self, loss, **_) -> "Metrics":
        return Metrics(float(loss), 1)

    def merge(self, other: "Metrics") -> "Metrics":
        return Metrics(self.total + other.total, self.count + other.count)

    def compute(self) -> dict:
        return {"loss": self.total / self.count if self.count else float("nan")}


class SimpleTrainer:
    """flaxdiff/trainer/simple_trainer.py:114-: the reference's trainer for ARBITRARY flax modules and loss
    functions (it differentiates them with jax.value_and_grad).  This engine has no autograd - the UNet's backward
    is an explicit program over libfdx kernels - so only the diffusion trainers exist; constructing this class
    says so instead of silently training something else."""

    def __init__(self, *args, **kwargs):
        raise FdxError("SimpleTrainer (generic model + loss_fn) is outside the supported hot path: this engine "
                       "trains flaxdiff_b200.models.simple_unet.Unet through GeneralDiffusionTrainer / DiffusionTrainer")
