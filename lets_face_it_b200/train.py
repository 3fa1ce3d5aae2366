"""Fused training step over the flat parameter buffer, with batch-sharded data parallelism.

Semantics of the reference's step (LetsFaceItGlow.training_step + configure_optimizers,
lets_face_it_glow.py:39-72, final_model.yaml: Adam lr 1e-5 betas (0.9, 0.9999), gradient_clip_val 20):
loss = mean_t mean_b NLL bits; backward; clip_grad_norm_(20); the optimizer `Optim.name` names (Adam, SGD or
RMSprop).  Here the whole step is a handful of stream-ordered launches with no host synchronisation: forward +
backward through the C ABI, one NCCL all-reduce of the flat fp32 gradient when world_size > 1 (the only exchange
the path has, SURVEY.md §8(e)), and a fused clip + update over the flat buffer.
"""
from __future__ import annotations

import inspect
import math

import torch

from . import _cabi as cabi

LN2 = math.log(2.0)

# configure_optimizers (lets_face_it_glow.py:61-72): Optim.name -> torch.optim class, built with Optim.args[name] and lr = hparams.lr
OPTIMIZERS = {"adam": torch.optim.Adam, "sgd": torch.optim.SGD, "rmsprop": torch.optim.RMSprop}
# torch.optim arguments whose non-default values the fused updates do not implement
_FIXED = {"adam": {"weight_decay": 0, "amsgrad": False}, "sgd": {}, "rmsprop": {}}
_OFF = ("maximize", "foreach", "fused", "capturable", "differentiable")


def choose_optimizer(hp, lr=None, betas=None, eps=None):
    """The optimizer of `configure_optimizers` for hparams `hp`: (name, keyword arguments of torch.optim.<name>, `lr`
    included, with every default filled in).  `lr` / `betas` / `eps` override hp.lr and Optim.args[name] as Trainer's
    arguments do.  Raises ValueError for an unknown name and (as torch does) for invalid values, TypeError for a keyword
    torch.optim does not accept, NotImplementedError for a value the fused update does not implement."""
    optim = hp.Optim
    name = optim.get("name")
    if name not in OPTIMIZERS:
        raise ValueError("Optim.name %r: the fused trainer runs %s" % (name, ", ".join(OPTIMIZERS)))
    args = dict((optim.get("args") or {}).get(name) or {})
    if betas is not None:
        args["betas"] = betas
    if eps is not None:
        args["eps"] = eps
    return name, optimizer_args(name, lr if lr is not None else hp.lr, args)


def optimizer_args(name, lr, args):
    """Validates `args` for torch.optim.<name> and returns them complete (torch's defaults filled in, `lr` included)."""
    cls = OPTIMIZERS[name]
    unknown = set(args) - (set(inspect.signature(cls.__init__).parameters) - {"self", "params", "lr"})
    if unknown:
        raise TypeError("%s got unexpected keyword arguments %s" % (cls.__name__, sorted(unknown)))
    for k, v in args.items():
        if (k in _OFF and v) or (k in _FIXED[name] and v != _FIXED[name][k]):
            raise NotImplementedError("%s: %s=%r is not implemented by the fused update" % (name, k, v))
    full = dict(cls([torch.zeros(1, requires_grad=True)], lr=float(lr), **args).defaults)  # torch's own value checks
    if "betas" in full:
        full["betas"] = tuple(float(b) for b in full["betas"])
    return full


def _buffer_names(name, args):
    """Flat state buffers of the optimizer, named as torch.optim names the per-parameter state."""
    if name == "adam":
        return ("exp_avg", "exp_avg_sq")
    if name == "sgd":
        return ("momentum_buffer",) if args["momentum"] != 0 else ()
    return ("square_avg",) + (("momentum_buffer",) if args["momentum"] > 0 else ()) + (("grad_avg",) if args["centered"] else ())


class _ScalarFeed:
    """A small device vector of per-step scalars, written from a ring of pinned host slots by stream-ordered copies (a slot
    is refilled only after the copy that last read it has run), so that a step never waits on the device."""

    def __init__(self, n, dev, slots=4):
        self.dev = torch.zeros(n, device=dev)
        self._host = [torch.zeros(n).pin_memory() for _ in range(slots)]
        self._host_ev = [torch.cuda.Event() for _ in range(slots)]
        self._i = 0

    def write(self, values):
        j = self._i
        self._i = (j + 1) % len(self._host)
        self._host_ev[j].synchronize()  # the copy that last used this pinned slot has been executed
        for i, v in enumerate(values):
            self._host[j][i] = v
        self.dev.copy_(self._host[j], non_blocking=True)
        self._host_ev[j].record()
        return self.dev


class Trainer:
    def __init__(self, model, lr=None, betas=None, eps=None, max_norm=None, process_group=None, dropout=True, probe_seed=1234):
        hp = model.hparams
        self.model = model
        self.eng = model.engine()
        self.optim, args = choose_optimizer(hp, lr, betas, eps)
        self.base_lr = float(args.pop("lr"))
        self.optim_args = args  # torch.optim keyword arguments besides lr
        self.lr = self.base_lr
        self.epoch = 0
        # configure_optimizers (lets_face_it_glow.py:61-72) returns get_scheduler(Optim.Schedule) (utils.py:65-82): StepLR per epoch
        sched = (hp.Optim.get("Schedule") or {}) if isinstance(getattr(hp, "Optim", None), dict) else {}
        self._sched_name = sched.get("name") or None
        self._sched_args = (sched.get("args") or {}).get(self._sched_name, {}) if self._sched_name else {}
        if self._sched_name not in (None, "step"):
            raise NotImplementedError("Unimplemented Scheduler!")  # utils.py:80 (multiplicative / lambda are unused by the shipped yamls)
        self.max_norm = float(max_norm if max_norm is not None else (hp.gradient_clip_val or 0))
        self.dropout = dropout
        dev = self.eng.theta.device
        n = self.eng.n_theta
        self.buffers = {k: torch.zeros(n, device=dev) for k in _buffer_names(self.optim, args)}
        self._buf_empty = True  # SGD: the momentum buffer holds no value yet (torch's first momentum step sets buf = g)
        self._feed = None       # per-step scalars of the SGD / RMSprop updates (Adam's eager launch takes them as arguments)
        self.gflat = self.eng.new_flat_grad()
        self.scratch = torch.zeros(2, device=dev)
        self.step_count = 0
        self.pg = process_group
        self.world = 1
        if torch.distributed.is_available() and torch.distributed.is_initialized():
            self.world = torch.distributed.get_world_size(process_group)
        # the probe decision of training_step must be the same on every rank (SURVEY.md section 8(e)): a generator of its own,
        # seeded identically everywhere, instead of the process-global `random` whose state differs between ranks
        import random
        self._probe_rng = random.Random(probe_seed) if self.world > 1 else random
        self._dnll = {}
        # LetsFaceItGlow.__init__ (lets_face_it_glow.py:28-36): state of the mismatched-NLL probe
        self.last_missmatched_nll = float("inf")
        self.missmatched_modalities, self.missmatched_nll_name = None, None
        if getattr(hp, "Train", None) and hp.Train.get("use_negative_nll_loss"):
            from .glow.utils import get_mismatched_modalities
            self.missmatched_modalities, self.missmatched_nll_name = get_mismatched_modalities(hp)
        # data parallel: the flow-step bucket of the gradient is reduced on a side stream while the encoder backward runs
        self.overlap = self.world > 1 and dev.type == "cuda"
        if self.overlap:
            self._side = torch.cuda.Stream(device=dev)
            self._ev = torch.cuda.Event()
            self._ev.record()  # creates the underlying cudaEvent
            self._bucket = flow_grad_range(self.eng.blocks)

    def broadcast_parameters(self, src=0):
        """Replicas start identical.  (The ActNorm data-dependent init is shared by `step` itself: it broadcasts rank 0's
        parameters right after the init, whatever the caller did before.)"""
        if self.world > 1:
            torch.distributed.broadcast(self.eng.theta, src, group=self.pg)

    def epoch_end(self):
        """StepLR(step_size, gamma) stepped once per epoch, as Lightning steps the scheduler `configure_optimizers` returns
        (lets_face_it_glow.py:61-72, utils.py:65-82; final_model.yaml: step_size 3, gamma 0.73)."""
        self.epoch += 1
        if self._sched_name == "step":
            self.lr = self.base_lr * float(self._sched_args.get("gamma", 0.1)) ** (self.epoch // int(self._sched_args["step_size"]))
        return self.lr

    def training_step(self, batch, masks=None):
        """`LetsFaceItGlow.training_step` (lets_face_it_glow.py:39-55) on the fused step: with `use_negative_nll_loss`, once
        the last mismatched NLL is positive, one step in ten (python `random`, as the reference) trains on a batch whose
        interlocutor modalities are shuffled across sequences (`derange_batch`) with the loss scaled by -0.1.  The `and`
        chain is evaluated in the reference's order, so `random.random()` is consumed on the same steps; the only host
        synchronisation is the read-back of the probe's NLL on those (10 %) steps.  Returns (loss, deranged)."""
        from .glow.utils import derange_batch

        hp = self.model.hparams
        if (hp.Train["use_negative_nll_loss"] and self.last_missmatched_nll > 0 and self._probe_rng.random() < 0.1
                and self.missmatched_modalities):
            loss = self.step(derange_batch(batch, self.missmatched_modalities), masks, loss_scale=-0.1)
            probe = loss.detach().clone()
            if self.world > 1:  # every rank must see the same `last_missmatched_nll`: mean over the global batch
                torch.distributed.all_reduce(probe, op=torch.distributed.ReduceOp.SUM, group=self.pg)
                probe /= self.world
            self.last_missmatched_nll = -float(probe)  # "Loss/missmatched_nll" (:51-52)
            return loss * -0.1, True
        return self.step(batch, masks), False

    def step(self, batch, masks=None, loss_scale=1.0):
        """One optimizer step on this rank's shard of sequences.  Returns the (device) loss of the shard (unscaled);
        `loss_scale` multiplies the loss the gradient is taken of (the -0.1 of the mismatched-NLL probe)."""
        scalars = self._advance()
        hyper = None
        if self.optim != "adam":
            if self._feed is None:
                self._feed = _ScalarFeed(len(scalars), self.eng.theta.device)
            hyper = self._feed.write(scalars)
        return self._step_body(batch, masks, loss_scale, hyper)

    def step_scalars(self):
        """The per-step scalars of the update at the CURRENT step count, in the layout its `_dev` entry reads:
        Adam (lr, 1 - beta1^step, sqrt(1 - beta2^step)) in double as torch.optim.Adam computes them; SGD (lr, 1 on the
        first momentum step else 0); RMSprop (lr,)."""
        if self.optim == "adam":
            b1, b2 = self.optim_args["betas"]
            return self.lr, 1.0 - b1 ** self.step_count, math.sqrt(1.0 - b2 ** self.step_count)
        if self.optim == "sgd":
            return self.lr, 1.0 if self._buf_empty else 0.0
        return (self.lr,)

    def _advance(self):
        """Counts one step and returns its scalars; the step that consumes them fills the momentum buffer."""
        self.step_count += 1
        scalars = self.step_scalars()
        self._buf_empty = False
        return scalars

    def _step_body(self, batch, masks, loss_scale, hyper):
        """The launches of one step.  `hyper` (device vector of `step_scalars()`, or None for Adam's eager launch): the
        per-step scalars are read on the device, so that the identical launch sequence can be captured once and replayed
        (GraphedStep)."""
        model = self.model
        eng = self.eng = model.engine()  # picks up a changed model.gemm_mode / a model moved to another device
        x0 = batch["p1_face"]
        B, T = x0.shape[0], x0.shape[1]
        Tp = T - eng.start_ts
        if masks is None and self.dropout and model.training:
            masks = model._masks(Tp, B, eng.theta.device)
        if model.training and not all(l.actnorm.inited for l in model.glow.flow.layers):
            model._ddi(eng, batch, masks)
            if self.world > 1:  # the init is data dependent: every replica takes rank 0's (the other shards' statistics are dropped)
                torch.distributed.broadcast(eng.theta, 0, group=self.pg)
        z, nll = eng.train_forward(batch, masks)
        key = (Tp, B, float(loss_scale))
        if key not in self._dnll:
            self._dnll[key] = torch.full((Tp, B), float(loss_scale) / (Tp * B), device=eng.theta.device)
        self.gflat.zero_()
        g = self.gflat[:eng.n_theta]
        if self.overlap:
            L = cabi.lib()
            L.lfi_set_grad_ready_event(self._ev.cuda_event)
            try:
                eng.train_backward(z, self._dnll[key], self.gflat)
            finally:
                L.lfi_set_grad_ready_event(None)
            lo, hi = self._bucket
            with torch.cuda.stream(self._side):
                self._side.wait_event(self._ev)  # recorded inside the backward call, before the encoder backward
                work = torch.distributed.all_reduce(g[lo:hi], op=torch.distributed.ReduceOp.SUM, group=self.pg, async_op=True)
            # ActNorm / 1x1-conv and encoder gradients are final only now.  The flat layout puts them behind the flow-step bucket
            # as one contiguous tail (engine.py: _layout), so this is ONE small all-reduce (2.4 MB) instead of two.
            for a0, a1 in ((0, lo), (hi, eng.n_theta)):
                if a1 > a0:
                    torch.distributed.all_reduce(g[a0:a1], op=torch.distributed.ReduceOp.SUM, group=self.pg)
            work.wait()
        else:
            eng.train_backward(z, self._dnll[key], self.gflat)
            allreduce_flat_gradient(g, self.world, self.pg)  # sum; averaged by grad_scale below
        loss = nll.mean() - eng.logdet_const() / LN2  # before the update: the parameter-only log-det term belongs to THIS step's theta
        self._update(g, hyper)
        return loss

    def _update(self, g, hyper):
        """The fused clip + optimizer update of the flat gradient `g` (two launches)."""
        L, eng, a, buf = cabi.lib(), self.eng, self.optim_args, self.buffers
        ptr = lambda k: buf[k].data_ptr() if k in buf else None
        if self.optim == "adam":
            (b1, b2), eps = a["betas"], a["eps"]
            if hyper is None:
                cabi.check(L.lfi_clip_adam(eng.theta.data_ptr(), g.data_ptr(), ptr("exp_avg"), ptr("exp_avg_sq"), eng.n_theta,
                                           self.lr, b1, b2, eps, self.max_norm, 1.0 / self.world,
                                           self.step_count, self.scratch.data_ptr(), cabi.stream_ptr()), "lfi_clip_adam")
            else:
                cabi.check(L.lfi_clip_adam_dev(eng.theta.data_ptr(), g.data_ptr(), ptr("exp_avg"), ptr("exp_avg_sq"), eng.n_theta,
                                               hyper.data_ptr(), b1, b2, eps, self.max_norm, 1.0 / self.world,
                                               self.scratch.data_ptr(), cabi.stream_ptr()), "lfi_clip_adam_dev")
        elif self.optim == "sgd":
            cabi.check(L.lfi_clip_sgd_dev(eng.theta.data_ptr(), g.data_ptr(), ptr("momentum_buffer"), eng.n_theta, hyper.data_ptr(),
                                          a["momentum"], a["dampening"], a["weight_decay"], int(a["nesterov"]), self.max_norm,
                                          1.0 / self.world, self.scratch.data_ptr(), cabi.stream_ptr()), "lfi_clip_sgd_dev")
        else:
            cabi.check(L.lfi_clip_rmsprop_dev(eng.theta.data_ptr(), g.data_ptr(), ptr("square_avg"), ptr("grad_avg"), ptr("momentum_buffer"),
                                              eng.n_theta, hyper.data_ptr(), a["alpha"], a["eps"], a["weight_decay"], a["momentum"],
                                              self.max_norm, 1.0 / self.world, self.scratch.data_ptr(), cabi.stream_ptr()),
                       "lfi_clip_rmsprop_dev")

    def graphed(self, batch, masks=None, warmup=3):
        """A `GraphedStep` over batches of the shape of `batch` (SURVEY.md section 8(f) rank 2)."""
        return GraphedStep(self, batch, masks, warmup)

    def grad_norm(self):
        """Global gradient norm of the last step (after the all-reduce average, before clipping)."""
        return torch.sqrt(self.scratch[0]) / self.world

    # ------------------------------------------------------------------ checkpoint / resume
    def state_dict(self):
        """Everything the next steps depend on besides the model's own parameters (kept apart, as Lightning keeps them):
        the optimizer name and arguments, its flat state buffers (cloned: the dict is a snapshot), the step count, epoch and
        learning rates, the mismatched-NLL probe's last value and, with world_size > 1, the probe generator's state (a single
        process draws from the caller's `random`, as the reference does)."""
        return {"optimizer": self.optim, "args": dict(self.optim_args),
                "buffers": {k: v.clone() for k, v in self.buffers.items()}, "buffers_empty": self._buf_empty,
                "step_count": self.step_count, "epoch": self.epoch, "base_lr": self.base_lr, "lr": self.lr,
                "last_missmatched_nll": self.last_missmatched_nll,
                "probe_rng": self._probe_rng.getstate() if self.world > 1 else None}

    def load_state_dict(self, sd):
        """Restores a `state_dict()`.  The buffers are copied into the existing ones, so a GraphedStep captured before the load
        continues from the loaded state."""
        if sd["optimizer"] != self.optim:
            raise ValueError("state of optimizer %r cannot load into a trainer running %r" % (sd["optimizer"], self.optim))
        args = optimizer_args(self.optim, sd["base_lr"], sd["args"])
        args.pop("lr")
        self._load_buffers(args, sd["buffers"].items())
        self._buf_empty = bool(sd["buffers_empty"])
        self.step_count, self.epoch = int(sd["step_count"]), int(sd["epoch"])
        self.base_lr, self.lr = float(sd["base_lr"]), float(sd["lr"])
        self.last_missmatched_nll = float(sd["last_missmatched_nll"])
        if self.world > 1 and sd.get("probe_rng") is not None:
            self._probe_rng.setstate(sd["probe_rng"])

    def _load_buffers(self, args, items):
        """Installs validated optimizer arguments and copies (name, flat tensor or [(offset, tensor)]) into the buffers."""
        if set(_buffer_names(self.optim, args)) != set(self.buffers):
            raise ValueError("%s state with buffers %s cannot load into a trainer whose arguments need %s"
                             % (self.optim, sorted(_buffer_names(self.optim, args)), sorted(self.buffers)))
        for k, src in items:
            if k not in self.buffers:
                raise ValueError("unexpected %s state buffer %r" % (self.optim, k))
            if torch.is_tensor(src):
                src = [(0, src)]
            for off, t in src:
                self.buffers[k][off:off + t.numel()].copy_(t.reshape(-1))
        self.optim_args = args

    def _param_offsets(self):
        """model.parameters(), each with its offset in the flat buffer (found by identity: the flat layout has its own order)."""
        where = {id(p): off for p, off, _ in self.model.engine()._views}
        params = list(self.model.parameters())
        missing = [i for i, p in enumerate(params) if id(p) not in where]
        if missing:
            raise RuntimeError("parameters %s of the model are not in the flat buffer" % missing)
        return [(p, where[id(p)]) for p in params]

    def optimizer_state_dict(self):
        """The optimizer state in the format of torch.optim.<Adam|SGD|RMSprop>.state_dict() over model.parameters() in that
        order (what a Lightning checkpoint stores under "optimizer_states"): built by a real torch optimizer, so keys, dtypes
        and devices are the installed torch's."""
        params = self._param_offsets()
        opt = OPTIMIZERS[self.optim]([p for p, _ in params], lr=self.lr, **self.optim_args)
        started = not self._buf_empty if self.optim == "sgd" else self.step_count > 0
        if started and (self.buffers or self.optim != "sgd"):
            for p, off in params:
                st = {} if self.optim == "sgd" else {"step": torch.tensor(float(self.step_count))}
                for k, b in self.buffers.items():
                    st[k] = b[off:off + p.numel()].view_as(p).clone()
                opt.state[p] = st
        return opt.state_dict()

    def load_optimizer_state_dict(self, sd):
        """Loads a torch.optim.<Adam|SGD|RMSprop>.state_dict() taken over model.parameters() (e.g. ckpt["optimizer_states"][0]
        of a Lightning run).  As torch does, the group's hyperparameters, lr included, come from the dict; Adam's and RMSprop's
        per-parameter `step` values must all be equal and become `step_count`."""
        groups = sd["param_groups"]
        params = self._param_offsets()
        if len(groups) != 1 or len(groups[0]["params"]) != len(params):
            raise ValueError("expected one parameter group over the model's %d parameters" % len(params))
        g = groups[0]
        hyper = {k: v for k, v in g.items() if k not in ("params", "lr", "initial_lr", "param_names")}
        try:
            args = optimizer_args(self.optim, g["lr"], hyper)
        except TypeError as e:
            raise ValueError("optimizer state does not belong to torch.optim.%s: %s" % (OPTIMIZERS[self.optim].__name__, e)) from None
        lr = args.pop("lr")
        state = [sd["state"].get(i, {}) for i in g["params"]]
        names = _buffer_names(self.optim, args)
        need = names + (() if self.optim == "sgd" else ("step",))
        have = [all(k in st for k in need) for st in state]
        empty = self.optim == "sgd" and not any(have)  # an SGD that has not stepped yet: no momentum buffers
        if not (all(have) or empty):
            i = have.index(False)
            raise ValueError("optimizer state of parameter %d lacks %s" % (i, [k for k in need if k not in state[i]]))
        if self.optim != "sgd":
            steps = {float(st["step"]) for st in state}
            if len(steps) != 1:
                raise ValueError("per-parameter step counts differ: %s" % sorted(steps))
            self.step_count = int(steps.pop())
        items = [] if empty else [(k, [(off, st[k]) for (_, off), st in zip(params, state)]) for k in names]
        self._load_buffers(args, items)
        if self.optim == "sgd":
            self._buf_empty = empty or not names
        self.lr = float(lr)
        if "initial_lr" in g:
            self.base_lr = float(g["initial_lr"])


class GraphedStep:
    """One training step (frame-dropout masks, forward + NLL, backward, clip, optimizer update: every launch of `Trainer.step`,
    side streams included) captured ONCE as a CUDA graph and replayed per step (SURVEY.md section 8(f) rank 2: "make the whole
    optimizer step graph-capturable").  What makes the step capturable: no host synchronisation anywhere in it, every buffer
    owned by the caller at a fixed address (grow-only workspace, flat theta / grad / optimizer state), and the only scalars that
    change from step to step - learning rate, Adam's bias corrections, SGD's first-momentum-step flag - read from device memory
    (`lfi_clip_adam_dev`, `lfi_clip_sgd_dev`, `lfi_clip_rmsprop_dev`).  The frame dropout draws from torch's CUDA generator,
    which torch advances per replay.  `Trainer.load_state_dict` copies into the captured buffers, so replays continue from a
    loaded state; a load that changes the optimizer arguments needs a new capture.

    `step(batch)` copies the batch into the captured input buffers, uploads the step's scalars (pinned, stream ordered) and
    replays; it returns the loss tensor of the captured step (overwritten by the next replay).  `warmup` eager steps run first
    (they ARE optimizer steps: ActNorm data-dependent init, workspace growth and the library's per-shape caches happen there).
    Single process only: with world_size > 1 the eager, stream-ordered `Trainer.step` is the path (its NCCL calls overlap the
    backward through events that are handed to the library per call)."""

    def __init__(self, trainer, batch, masks=None, warmup=3):
        if trainer.world > 1:
            raise NotImplementedError("GraphedStep: single-process only; use Trainer.step under torch.distributed")
        tr = self.tr = trainer
        dev = tr.eng.theta.device
        if dev.type != "cuda":
            raise RuntimeError("GraphedStep needs a CUDA device (no CPU path)")
        self.static = {k: v.to(dev).float().contiguous().clone() for k, v in batch.items() if torch.is_tensor(v)}
        self.masks = masks
        self._feed = _ScalarFeed(len(tr.step_scalars()), dev)
        self.hyper = self._feed.dev
        self._args = dict(tr.optim_args)  # captured as launch arguments
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            for _ in range(max(int(warmup), 1)):
                tr.step(self.static, masks)
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize(dev)
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.loss = tr._step_body(self.static, masks, 1.0, self.hyper)

    def step(self, batch=None):
        tr = self.tr
        if batch is not None:
            for k, dst in self.static.items():
                src = batch[k]
                if src.data_ptr() != dst.data_ptr():
                    dst.copy_(src, non_blocking=True)
        if tr.optim_args != self._args:
            raise RuntimeError("GraphedStep: the optimizer arguments changed since the capture (%s -> %s); capture a new one"
                               % (self._args, tr.optim_args))
        self._feed.write(tr._advance())
        self.graph.replay()
        return self.loss


class HostFeed:
    """End-to-end driver over host batches (what a DataLoader with pinned memory hands to `LetsFaceItGlow.training_step`):
    every step's inputs are copied host -> device on a copy stream into one of two device buffers while the previous step
    computes, and every step's loss is read back (device -> host) one step late, so that neither the copy nor the read-back
    leaves the GPU idle.  `step(host_batch)` returns the loss (python float) of the PREVIOUS call (None on the first);
    `flush()` returns the last one."""

    def __init__(self, trainer):
        self.tr = trainer
        dev = trainer.eng.theta.device
        self.dev = dev
        self.copy_stream = torch.cuda.Stream(device=dev)
        self.bufs = [None, None]
        self.copied = [torch.cuda.Event(), torch.cuda.Event()]
        self.consumed = [torch.cuda.Event(), torch.cuda.Event()]
        self.i = 0
        self.pending = None  # (pinned host scalar, event) of the previous step's loss
        self._loss_host = [torch.empty(1, dtype=torch.float32).pin_memory() for _ in range(2)]
        self._loss_ev = [torch.cuda.Event(), torch.cuda.Event()]

    def step(self, host_batch, masks=None):
        j = self.i & 1
        cur = torch.cuda.current_stream(self.dev)
        with torch.cuda.stream(self.copy_stream):
            if self.i >= 2:
                self.copy_stream.wait_event(self.consumed[j])  # the step that last read this buffer is done
            if self.bufs[j] is None or any(self.bufs[j][k].shape != v.shape for k, v in host_batch.items()):
                self.bufs[j] = {k: torch.empty(v.shape, dtype=torch.float32, device=self.dev) for k, v in host_batch.items()}
            for k, v in host_batch.items():
                self.bufs[j][k].copy_(v, non_blocking=True)
            self.copied[j].record(self.copy_stream)
        cur.wait_event(self.copied[j])
        loss = self.tr.step(self.bufs[j], masks)
        self.consumed[j].record(cur)
        self._loss_host[j].copy_(loss.detach().reshape(1), non_blocking=True)
        self._loss_ev[j].record(cur)
        prev = self.flush() if self.pending is not None else None
        self.pending = j
        self.i += 1
        return prev

    def flush(self):
        """Loss of the most recent step whose read-back has not been returned yet."""
        if self.pending is None:
            return None
        j, self.pending = self.pending, None
        self._loss_ev[j].synchronize()
        return float(self._loss_host[j][0])


class ResidentFeed:
    """End-to-end driver over an HBM-resident corpus (`lets_face_it_b200.data.ResidentWindows`, SURVEY.md section 8(f) rank 4):
    per step the host sends only the window table entries of the batch (8 bytes per sequence instead of 55 KB), the batch is
    gathered on the device, and the loss is read back one step late as in `HostFeed`."""

    def __init__(self, trainer, windows):
        self.tr, self.ds = trainer, windows
        self.bufs = {}
        self.pending = None
        self._loss_host = [torch.empty(1, dtype=torch.float32).pin_memory() for _ in range(2)]
        self._loss_ev = [torch.cuda.Event(), torch.cuda.Event()]
        self.i = 0

    def step(self, index, masks=None):
        j = self.i & 1
        batch = self.ds.batch(index, out=self.bufs)
        loss = self.tr.step(batch, masks)
        self._loss_host[j].copy_(loss.detach().reshape(1), non_blocking=True)
        self._loss_ev[j].record(torch.cuda.current_stream(self.ds.device))
        prev = self.flush() if self.pending is not None else None
        self.pending = j
        self.i += 1
        return prev

    def flush(self):
        if self.pending is None:
            return None
        j, self.pending = self.pending, None
        self._loss_ev[j].synchronize()
        return float(self._loss_host[j][0])


def allreduce_flat_gradient(g, world, group=None):
    """The one exchange of the path (SURVEY.md §8(e)): SUM all-reduce of the flat fp32 gradient over the ranks.
    The mean over the global batch is restored by `grad_scale = 1/world` in the fused clip+Adam (every rank holds an
    equal shard and the reference loss is a batch mean, models.py:555), so clipping sees the global-batch gradient."""
    if world > 1:
        torch.distributed.all_reduce(g, op=torch.distributed.ReduceOp.SUM, group=group)
    return g


# flat-buffer blocks whose gradients are final before the encoder backward (engine.py: _STEP_BLOCKS_F, contiguous)
_FLOW_BUCKET = ("wc", "bc", "w_ih", "b_ih", "w_hh", "b_hh", "wf", "bf", "lf")


def flow_grad_range(blocks):
    """[lo, hi) of the flat gradient covered by the flow-step weight blocks (`blocks`: name -> (offset, numel per step,
    steps), Engine.blocks).  The blocks must be adjacent in the flat layout (only alignment padding between them)."""
    spans = sorted((blocks[n][0], blocks[n][0] + blocks[n][1] * blocks[n][2]) for n in _FLOW_BUCKET if n in blocks)
    if not spans:
        return 0, 0
    lo, hi = spans[0][0], spans[-1][1]
    inside = {n for n, (o, m, k) in blocks.items() if lo <= o < hi}
    if inside != {n for n in _FLOW_BUCKET if n in blocks}:
        raise RuntimeError("flat layout changed: blocks %s lie inside the flow-step bucket" % sorted(inside - set(_FLOW_BUCKET)))
    return lo, hi


def shard_batch(batch, rank, world):
    """Contiguous, equal shards of the sequence batch (SURVEY.md §8(e)); B must divide evenly so the mean over
    the global batch equals the mean of the per-rank means."""
    out = {}
    for k, v in batch.items():
        B = v.shape[0]
        if B % world:
            raise ValueError("batch size %d is not divisible by world size %d" % (B, world))
        n = B // world
        out[k] = v[rank * n:(rank + 1) * n]
    return out
