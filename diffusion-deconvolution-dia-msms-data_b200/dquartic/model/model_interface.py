"""Training harness — drop-in for /root/reference/dquartic/model/model_interface.py (ModelInterface 238-1150,
WarmupLR_Scheduler 64-194, CallbackHandler 196-236) on B200.

Kept from the reference: the public method names and arguments, epoch-level warm-up + half-cosine LR schedule,
grad-clip 10.0 + AdamW(lr, betas (0.9, 0.999), eps 1e-8, weight_decay 0.01), checkpoint dictionary keys
(`epoch, model_state_dict, optimizer_state_dict, scheduler_state_dict, best_loss`) and file naming, the
0.5/0.5 mixing of the two drawn samples, `predict` returning dicts `{ms2_1, ms1_1, mixture, pred}`.

New: the optimizer step is three fused kernels over the flat parameter buffer (`FusedAdamW`), optionally keeping an
exponential moving average of the weights in the same pass (`ema_decay`, `ema_weights()`); a batch larger than
`micro_batch` is processed by gradient accumulation; under `torch.distributed` the batch is sharded by sample and
the flat gradient is summed over the ranks in buckets (the four 300 M-parameter mid-block ranges are launched as soon as
the mid-stage backward has produced them, overlapping the long down-path backward).  Those ranges (99 % of the
parameters) are REDUCE-SCATTERED: each rank keeps Adam moments for, and updates, 1 / world-size of them and the updated
pieces are all-gathered in place (ZeRO-1); 1 / world-size is folded into the clip coefficient; rank 0 writes checkpoints.
Plotting / wandb tables (reference 669-976, 1152-1242) are out of scope (SURVEY.md §2).
"""
import contextlib
import functools
import math
import os
from typing import List

import numpy as np
import torch
from torch.optim.lr_scheduler import LambdaLR

from .. import _native as N


# ------------------------------------------------------------------------------------------------ LR schedule
class LR_SchedulerInterface(object):
    def __init__(self, optimizer, **kwargs):
        raise NotImplementedError

    def step(self, epoch: int, loss: float):
        raise NotImplementedError

    def get_last_lr(self) -> List[float]:
        raise NotImplementedError


def _warmup_cosine_lambda(current_step, *, num_warmup_steps, num_training_steps, num_cycles):
    """reference model_interface.py:149-155."""
    if current_step < num_warmup_steps:
        return float(current_step + 1) / float(max(1, num_warmup_steps))
    progress = float(current_step - num_warmup_steps) / float(max(1, num_training_steps - num_warmup_steps))
    return max(1e-10, 0.5 * (1.0 + math.cos(math.pi * float(num_cycles) * 2.0 * progress)))


class WarmupLR_Scheduler(LR_SchedulerInterface):
    """Linear warm-up then half-cosine decay, stepped once per EPOCH (reference 64-194)."""

    def __init__(self, optimizer, num_warmup_steps: int, num_training_steps: int, num_cycles: float = 0.5,
                 last_epoch: int = -1, **kwargs):
        self.optimizer = optimizer
        self.lambda_lr = self.get_cosine_schedule_with_warmup(optimizer, num_warmup_steps, num_training_steps,
                                                              num_cycles=num_cycles, last_epoch=last_epoch)

    def step(self, epoch: int = None, loss=None):
        return self.lambda_lr.step()

    def get_last_lr(self) -> List[float]:
        return self.lambda_lr.get_last_lr()

    def _get_cosine_schedule_with_warmup_lr_lambda(self, current_step, *, num_warmup_steps, num_training_steps,
                                                   num_cycles):
        return _warmup_cosine_lambda(current_step, num_warmup_steps=num_warmup_steps,
                                     num_training_steps=num_training_steps, num_cycles=num_cycles)

    def get_cosine_schedule_with_warmup(self, optimizer, num_warmup_steps, num_training_steps, num_cycles=0.5,
                                        last_epoch=-1):
        fn = functools.partial(_warmup_cosine_lambda, num_warmup_steps=num_warmup_steps,
                               num_training_steps=num_training_steps, num_cycles=num_cycles)
        return LambdaLR(optimizer, fn, last_epoch)


class CallbackHandler:
    """No-op hooks; `epoch_callback` returning False stops training (reference 196-236)."""

    def epoch_callback(self, epoch: int, epoch_loss: float) -> bool:
        return True

    def batch_callback(self, batch: int, batch_loss: float):
        pass


# ------------------------------------------------------------------------------------------------ optimizer
class FusedAdamW(torch.optim.Optimizer):
    """AdamW over the flat parameter buffer of a B200 `UNet1d`: grad-norm, clip coefficient and the update are
    three kernels (dq_sumsq, dq_clip_coef, dq_adamw), no host synchronisation.  `state_dict()` /
    `load_state_dict()` speak torch.optim.AdamW's per-parameter format so reference checkpoints round-trip.

    Data parallel: the gradient buffer holds the SUM over ranks; `grad_scale = 1 / world-size` is folded into the clip
    coefficient (no averaging pass).  Sharded mode (`set_sharding`): the ranges listed there were reduce-scattered, this
    rank owns piece `rank` of each of them and keeps Adam moments for its pieces only (1 / world-size of the state,
    1 / world-size of the update traffic); the small rest of the buffer is replicated and updated by every rank; the
    updated pieces are all-gathered in place into the flat parameter buffer.

    `ema_decay` (0 < ema_decay < 1, default None: off) keeps an exponential moving average of the weights, updated in
    the same pass as AdamW (dq_adamw_ema) and laid out like the Adam moments (sharded mode: this rank's pieces plus the
    replicated rest).  Update k (from 0) uses the decay min(ema_decay, (1 + k) / (10 + k)).  `swap_ema()` exchanges
    it with the live weights; `ema_state_dict()` returns it in the model's state-dict format."""

    def __init__(self, net, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=1e-2, ema_decay=None):
        if ema_decay is not None and not 0.0 < float(ema_decay) < 1.0:
            raise ValueError(f"ema_decay must be None or in (0, 1), got {ema_decay}")
        self.net = net
        params = list(net.parameters())
        defaults = dict(lr=lr, betas=betas, eps=eps, weight_decay=weight_decay, amsgrad=False, maximize=False,
                        foreach=None, capturable=False, differentiable=False, fused=None)
        super().__init__(params, defaults)
        self._m = None
        self._v = None
        self._step = 0
        self._scratch = None
        self.last_grad_norm = None
        self._shard = None      # (rank, world, [(offset, numel)]) of the reduce-scattered ranges
        self._segments = None   # [(flat offset, numel, state offset)] this rank updates
        self._full_state = None
        self.ema_decay = None if ema_decay is None else float(ema_decay)
        self._ema = None            # EMA of the weights, same layout as _m / _v
        self.ema_updates = 0        # EMA updates so far (k of the decay warm-up)
        self._ema_swapped = False   # swap_ema(): the network holds the EMA, _ema the live weights

    @staticmethod
    def ema_beta(ema_decay, k):
        """Decay of EMA update k (counting from 0): a short warm-up so that the average forgets the initial weights."""
        return min(ema_decay, (1.0 + k) / (10.0 + k))

    # ---- layout of the state this rank keeps
    def set_sharding(self, rank, world, ranges):
        """Call before the first step.  `ranges`: sorted, disjoint (offset, numel) with numel % world == 0."""
        if self._m is not None:
            raise RuntimeError("set_sharding must be called before the optimizer state exists")
        self._shard = (int(rank), int(world), [(int(o), int(n)) for o, n in sorted(ranges)]) if world > 1 and ranges else None

    def _build_segments(self):
        n = self.net.n_trainable_flat
        if self._shard is None:
            return [(0, n, 0)]
        rank, world, ranges = self._shard
        segs, pos, so = [], 0, 0
        for (o, cnt) in ranges:
            if o > pos:                       # replicated gap before the sharded range
                segs.append((pos, o - pos, so)); so += o - pos
            k = cnt // world
            segs.append((o + rank * k, k, so)); so += k
            pos = o + cnt
        if pos < n:
            segs.append((pos, n - pos, so)); so += n - pos
        return segs

    def _ensure_state(self):
        flat = self.net.flat_params()
        if self._m is None or self._m.device != flat.device:
            self._segments = self._build_segments()
            total = sum(c for _, c, _ in self._segments)
            self._m = torch.zeros(total, dtype=torch.float32, device=flat.device)
            self._v = torch.zeros(total, dtype=torch.float32, device=flat.device)
            self._sumsq = torch.zeros(1, dtype=torch.float64, device=flat.device)
            self._coef = torch.zeros(2, dtype=torch.float32, device=flat.device)
            if self.ema_decay is not None:
                self._ema = torch.empty(total, dtype=torch.float32, device=flat.device)
                self.reset_ema()

    @torch.no_grad()
    def reset_ema(self):
        """Start the EMA over at the current weights (update count 0)."""
        if self._ema_swapped:
            raise RuntimeError("reset_ema() inside ema_weights()")
        self._ensure_state()
        flat = self.net.flat_params()
        for (o, cnt, so) in self._segments:
            self._ema[so:so + cnt].copy_(flat[o:o + cnt])
        self.ema_updates = 0
        self._full_state = None

    def zero_grad(self, set_to_none: bool = False):
        self.net.zero_grad()

    @torch.no_grad()
    def step(self, closure=None, max_grad_norm=None, grad_scale=1.0, defer_gather=False):
        """`defer_gather` (sharded mode): leave the parameter all-gathers in flight on the NCCL stream; the network waits
        for them right before its mid stage (`UNet1d.sync_params`), so they overlap the next step's down path."""
        if self._ema_swapped:
            raise RuntimeError("FusedAdamW.step() while the network holds the EMA weights (inside ema_weights())")
        self._ensure_state()
        net = self.net
        g = net.flat_grads()
        p = net.flat_params()
        grp = self.param_groups[0]
        lr, (b1, b2), eps, wd = grp["lr"], grp["betas"], grp["eps"], grp["weight_decay"]
        self._step += 1
        coef = None
        sharded = self._shard is not None
        if max_grad_norm is not None or grad_scale != 1.0:
            self._sumsq.zero_()
            if sharded:
                # every element of the buffer counted exactly once over the ranks: own pieces everywhere, the replicated
                # rest on rank 0 only; then one 8-byte all-reduce
                rank, world, ranges = self._shard
                owned = {(o + rank * (cnt // world)) for o, cnt in ranges}
                for (o, cnt, _) in self._segments:
                    if o in owned or rank == 0:
                        N.call("dq_sumsq", g[o:o + cnt], cnt, self._sumsq)
                torch.distributed.all_reduce(self._sumsq)
            else:
                N.call("dq_sumsq", g, net.n_trainable_flat, self._sumsq)
            big = 3.0e38 if max_grad_norm is None else float(max_grad_norm)
            N.call("dq_clip_coef", self._sumsq, big, float(grad_scale), self._coef)
            coef = self._coef
            self.last_grad_norm = self._coef[0:1]
        bc1 = 1.0 - b1 ** self._step
        bc2 = 1.0 - b2 ** self._step
        ema = self._ema
        if ema is not None:
            ema_w = 1.0 - self.ema_beta(self.ema_decay, self.ema_updates)   # rounded to fp32 by the call
            self.ema_updates += 1
        for (o, cnt, so) in self._segments:
            if ema is None:
                N.call("dq_adamw", p[o:o + cnt], g[o:o + cnt], self._m[so:so + cnt], self._v[so:so + cnt], cnt, coef, lr,
                       b1, b2, eps, wd, lr / bc1, math.sqrt(bc2))
            else:
                N.call("dq_adamw_ema", p[o:o + cnt], g[o:o + cnt], self._m[so:so + cnt], self._v[so:so + cnt],
                       ema[so:so + cnt], cnt, coef, lr, b1, b2, eps, wd, lr / bc1, math.sqrt(bc2), ema_w)
        if sharded:
            works = self._gather_params(p)
            if defer_gather and hasattr(net, "sync_params"):
                net.__dict__.setdefault("_pending_param_works", []).extend(works)
            else:
                for w in works:
                    w.wait()
        self._full_state = None
        net.mark_params_modified()

    def _gather_params(self, p):
        """Sharded mode: all-gather every rank's piece of the sharded ranges into the flat parameter buffer, in place."""
        rank, world, ranges = self._shard
        works = []
        for (o, cnt) in ranges:
            k = cnt // world
            works.append(torch.distributed.all_gather_into_tensor(p[o:o + cnt], p[o + rank * k:o + (rank + 1) * k],
                                                                  async_op=True))
        return works

    # ---- weight EMA ---------------------------------------------------------------------------------------
    def _require_ema(self):
        if self.ema_decay is None:
            raise RuntimeError("this FusedAdamW keeps no weight EMA (ema_decay=None)")
        self._ensure_state()

    @torch.no_grad()
    def swap_ema(self):
        """Exchange the EMA and the live weights in the network's flat parameter buffer (sharded mode: a collective, every
        rank; the swapped pieces are all-gathered).  Calling it twice restores the live weights bit for bit."""
        self._require_ema()
        net = self.net
        p = net.flat_params()
        for (o, cnt, so) in self._segments:
            N.call("dq_swap", p[o:o + cnt], self._ema[so:so + cnt], cnt)
        if self._shard is not None:
            for w in self._gather_params(p):
                w.wait()
        self._ema_swapped = not self._ema_swapped
        net.mark_params_modified()   # the bf16 GEMM operands are recast from the new weights

    def _full_ema(self):
        """EMA over the trainable flat range.  Sharded mode: needs `gather_state()` beforehand, unless the network holds
        the EMA (swap_ema), whose buffer then has it in full on every rank."""
        n = self.net.n_trainable_flat
        if self._ema_swapped:
            return self.net.flat_params()[:n]
        if self._shard is None:
            return self._ema
        if self._full_state is None or len(self._full_state) < 3:
            raise RuntimeError("sharded FusedAdamW: call gather_state() on every rank before ema_state_dict()")
        return self._full_state[2]

    @torch.no_grad()
    def ema_state_dict(self, device=None):
        """The EMA in the format of `UNet1d.state_dict()` (same names, shapes and order; the non-trainable rotary
        frequencies are the live model's), as copies on `device` (default: the EMA's device)."""
        self._require_ema()
        net = self.net
        full = self._full_ema()
        out = {}
        for name in net.state_dict(keep_vars=True):
            par = net._params[name]
            src = net._view(full, name) if par.requires_grad else par.detach()
            dst = torch.empty(src.shape, dtype=src.dtype, device=src.device if device is None else device)
            out[name] = dst.copy_(src)
        return out

    @torch.no_grad()
    def load_ema_state_dict(self, sd, updates):
        """Inverse of `ema_state_dict()`; `updates` is the EMA update count to resume from.  Sharded mode: this rank
        keeps its own pieces and the replicated rest."""
        self._require_ema()
        if self._ema_swapped:
            raise RuntimeError("load_ema_state_dict() inside ema_weights()")
        net = self.net
        if self._shard is None:
            full = self._ema
        else:
            full = torch.zeros(net.n_trainable_flat, dtype=torch.float32, device=self._ema.device)
        for name, par in net._params.items():
            if par.requires_grad:
                net._view(full, name).copy_(sd[name])
        if self._shard is not None:
            for (o, cnt, so) in self._segments:
                self._ema[so:so + cnt].copy_(full[o:o + cnt])
        self.ema_updates = int(updates)
        self._full_state = None

    # ---- full-size moments (checkpoints) ----------------------------------------------------------------
    def _full_moments(self):
        """(m, v) over the whole flat buffer.  Sharded mode: needs `gather_state()` (a collective) beforehand."""
        if self._shard is None:
            return self._m, self._v
        if self._full_state is None:
            raise RuntimeError("sharded FusedAdamW: call gather_state() on every rank before state_dict()")
        return self._full_state[:2]

    @torch.no_grad()
    def gather_state(self):
        """Collective (every rank): assemble the full Adam moments (and the EMA, unless the network holds it) from the
        shards, for `state_dict()` / `ema_state_dict()`."""
        self._ensure_state()
        if self._shard is None:
            return
        rank, world, ranges = self._shard
        n = self.net.n_trainable_flat
        srcs = (self._m, self._v) + ((self._ema,) if self._ema is not None and not self._ema_swapped else ())
        full = [torch.zeros(n, dtype=torch.float32, device=self._m.device) for _ in srcs]
        for (o, cnt, so) in self._segments:
            for f, src in zip(full, srcs):
                f[o:o + cnt].copy_(src[so:so + cnt])
        for (o, cnt) in ranges:
            k = cnt // world
            for f in full:
                torch.distributed.all_gather_into_tensor(f[o:o + cnt], f[o + rank * k:o + (rank + 1) * k].clone())
        self._full_state = tuple(full)

    # torch.optim.AdamW-compatible (de)serialisation -------------------------------------------------------
    def state_dict(self):
        self._ensure_state()
        net = self.net
        state = {}
        names = list(net._params.keys())
        if self._step > 0:
            m_full, v_full = self._full_moments()
        for idx, name in enumerate(names):
            if not net._params[name].requires_grad or self._step == 0:
                continue
            state[idx] = {"step": torch.tensor(float(self._step)),
                          "exp_avg": net._view(m_full, name).clone(),
                          "exp_avg_sq": net._view(v_full, name).clone()}
        groups = [{k: v for k, v in self.param_groups[0].items() if k != "params"}]
        groups[0]["params"] = list(range(len(names)))
        return {"state": state, "param_groups": groups}

    def load_state_dict(self, sd):
        self._ensure_state()
        net = self.net
        names = list(net._params.keys())
        n = net.n_trainable_flat
        if self._shard is None:
            m_full, v_full = self._m, self._v
            m_full.zero_()
            v_full.zero_()
        else:
            m_full = torch.zeros(net.flat_params().numel(), dtype=torch.float32, device=self._m.device)
            v_full = torch.zeros_like(m_full)
        step = 0
        for idx, st in sd["state"].items():
            name = names[int(idx)]
            net._view(m_full, name).copy_(st["exp_avg"])
            net._view(v_full, name).copy_(st["exp_avg_sq"])
            step = max(step, int(float(st["step"])))
        if self._shard is not None:
            for (o, cnt, so) in self._segments:
                self._m[so:so + cnt].copy_(m_full[o:o + cnt])
                self._v[so:so + cnt].copy_(v_full[o:o + cnt])
        self._step = step
        self._full_state = None
        for k, v in sd["param_groups"][0].items():
            if k != "params":
                self.param_groups[0][k] = v


# ------------------------------------------------------------------------------------------------ harness
class ModelInterface(object):
    def __init__(self, device=None, min_pred_value: float = 0.0, **kwargs):
        self.model: torch.nn.Module = None
        self.optimizer = None
        self.model_params: dict = {}
        self.min_pred_value = min_pred_value
        self.lr_scheduler_class = WarmupLR_Scheduler
        self.callback_handler = CallbackHandler()
        self.device = device if device is not None else torch.device("cuda" if torch.cuda.is_available() else "cpu")
        self.ms1_loss_weight = None
        self.use_wandb = False
        # B200 additions
        self.micro_batch = None       # samples per forward/backward pass (None: chosen from the free HBM, <= 64)
        self.max_grad_norm = 10.0     # reference model_interface.py:1121
        self.grad_bucket_elems = 64 * 1024 * 1024
        self.ema_decay = None         # weight EMA kept by the fused optimizer (None: off); see ema_weights()
        self.validation = None        # a dquartic.utils.validation.ValidationSet (None: off); see validate()
        self.val_history = []         # one dict per validated epoch

    def __repr__(self):
        return (f"{self.__class__.__name__} with {self.model.__class__.__name__} model with "
                f"{self.get_parameter_num()} parameters on {self.device}")

    # ---------------------------------------------------------------------------------------- public
    def build(self, model_class, **kwargs):
        self.model = model_class  # an INSTANCE, as in the reference (model_interface.py:298-299)
        self._init_for_training()

    def get_parameter_num(self):
        return np.sum([p.numel() for p in self.model.parameters()])

    def train_step(self, x_0, ms2_cond=None, ms1_cond=None, noise=None, ms1_loss_weight=0.0):
        raise NotImplementedError

    def sample(self, x_t, ms2_cond=None, ms1_cond=None, num_steps=1000, sampler="reference"):
        raise NotImplementedError

    def _ckpt_latest(self, checkpoint_path):
        return f"{os.path.dirname(checkpoint_path)}{os.path.sep}dquartic_latest_checkpoint.ckpt"

    def _is_rank0(self):
        return not (torch.distributed.is_available() and torch.distributed.is_initialized()) or \
            torch.distributed.get_rank() == 0

    def _run_epochs(self, dataloader, num_epochs, lr_scheduler, use_wandb, log_every_n_epochs, checkpoint_path):
        start_epoch, best_loss, lr_scheduler = self.load_checkpoint(lr_scheduler, self._ckpt_latest(checkpoint_path),
                                                                    self.device)
        best_epoch = start_epoch
        vset = self.validation
        if start_epoch > 0:
            # resumed run: do not replay the (t, noise) stream of the first epochs; every rank keeps its own stream
            rank = torch.distributed.get_rank() if self._dist_on() else 0
            torch.manual_seed(1234 + rank + 7919 * start_epoch)
        for epoch in range(start_epoch, num_epochs):
            if hasattr(dataloader, "dataset") and hasattr(dataloader.dataset, "reset_epoch"):
                dataloader.dataset.reset_epoch()
            batch_loss = self._train_one_epoch(epoch, dataloader)
            avg = float(np.mean(batch_loss))
            if lr_scheduler is not None:
                lr_scheduler.step(epoch, avg)
                lr_now = lr_scheduler.get_last_lr()[0]
            else:
                lr_now = self.optimizer.param_groups[0]["lr"]
            if use_wandb and self._is_rank0():
                import wandb
                wandb.log({"epoch": epoch, "train/loss": avg, "learning_rate": lr_now})
            # with validation the held-out loss (the EMA's when the EMA is on) selects the best checkpoint, and only
            # epochs that ran it can become the best; without it, the epoch-mean training loss does
            metric, val_kw = avg, {}
            if vset is not None:
                metric = self._validate_epoch(epoch, use_wandb) if vset.due(epoch) else None
                val_kw = {"val_loss": metric}
            if isinstance(self.optimizer, FusedAdamW):
                self.optimizer.gather_state()   # sharded optimizer: collective, every rank (no-op otherwise)
            better = metric is not None and metric < best_loss
            if better:
                best_loss, best_epoch = metric, epoch + 1
            if self._is_rank0():
                print(f"[Training] Epoch={epoch+1}, lr={lr_now}, loss={avg}")
                self.save_checkpoint(lr_scheduler, epoch, avg if vset is None else best_loss,
                                     self._ckpt_latest(checkpoint_path), **val_kw)
                if better:
                    self.save_checkpoint(lr_scheduler, epoch, best_loss, checkpoint_path, **val_kw)
            if use_wandb and (epoch == 0 or epoch % log_every_n_epochs == 0) and self._is_rank0():
                # the reference logs a plotted prediction here (model_interface.py:440-448); plotting is out of scope of
                # this build, so the training loop must not die on it (a raise here would kill rank 0 after the first
                # epoch and leave the other ranks blocked in NCCL): warn once, keep training
                try:
                    self.log_single_prediction(best_epoch, best_loss, dataloader, num_steps=[100, 500, 1000],
                                               path=f"{os.path.dirname(checkpoint_path)}{os.path.sep}")
                except (ImportError, NotImplementedError) as e:
                    if not getattr(self, "_warned_no_plot", False):
                        self._warned_no_plot = True
                        print(f"Warning: prediction plots are not logged ({e}); scalar metrics still go to wandb")
            if not self.callback_handler.epoch_callback(epoch=epoch, epoch_loss=avg):
                print(f"Training stopped at epoch {epoch}")
                break
        if self._is_rank0():
            print(f"Best model checkpoint saved at epoch {best_epoch} with loss: {best_loss:.6f}")

    def _validate_epoch(self, epoch, use_wandb):
        """`validate` on the live weights and, with the EMA on, inside `ema_weights()` (every rank); records, prints and
        logs them.  Returns the selection metric: the EMA's val_loss when the EMA is on, else the live one."""
        vset = self.validation
        live = self.validate(vset)
        rec = {"epoch": epoch + 1, "val_loss": live["val_loss"], "loss_by_band": live["loss_by_band"]}
        metric = live["val_loss"]
        if self._ema_on():
            with self.ema_weights():
                ema = self.validate(vset)
            rec.update(ema_val_loss=ema["val_loss"], ema_loss_by_band=ema["loss_by_band"])
            metric = ema["val_loss"]
        self.val_history.append(rec)
        if self._is_rank0():
            ema_txt = f", ema_val_loss={rec['ema_val_loss']}" if "ema_val_loss" in rec else ""
            print(f"[Validation] Epoch={epoch + 1}, val_loss={rec['val_loss']}{ema_txt}")
            if use_wandb:
                import wandb
                log = {"epoch": epoch, "val/loss": rec["val_loss"]}
                log.update({f"val/loss_t{t}": float(v) for t, v in zip(vset.bands, rec["loss_by_band"])})
                if "ema_val_loss" in rec:
                    log["val_ema/loss"] = rec["ema_val_loss"]
                wandb.log(log)
        return metric

    def train_with_warmup(self, dataloader, num_epochs, num_warmup_steps=5, learning_rate=1e-4, use_wandb=True,
                          log_every_n_epochs=100, checkpoint_path="best_model.ckpt"):
        self._prepare_training(learning_rate)
        lr_scheduler = self._get_lr_schedule_with_warmup(num_warmup_steps, num_epochs)
        self.model.train()
        self._run_epochs(dataloader, num_epochs, lr_scheduler, use_wandb, log_every_n_epochs, checkpoint_path)

    def train(self, dataloader, batch_size, epochs, warmup_epochs: int = 5, learning_rate: float = 1e-4,
              use_wandb: bool = False, checkpoint_path: str = "best_model.ckpt", **kwargs):
        if self._is_rank0():
            print(f"Info: Training {self!r}")
        if warmup_epochs > 0:
            self.train_with_warmup(dataloader, epochs, num_warmup_steps=warmup_epochs, learning_rate=learning_rate,
                                   use_wandb=use_wandb, checkpoint_path=checkpoint_path, **kwargs)
        else:
            self._prepare_training(learning_rate, **kwargs)
            self._run_epochs(dataloader, epochs, None, use_wandb, 100, checkpoint_path)

    def load_checkpoint(self, scheduler, checkpoint_path, device):
        if os.path.exists(checkpoint_path):
            print(f"Loading checkpoint from {checkpoint_path}...")
            checkpoint = torch.load(checkpoint_path, map_location=device, weights_only=False)
            self.model.load_state_dict(checkpoint["model_state_dict"])
            if self.optimizer is not None:
                self.optimizer.load_state_dict(checkpoint["optimizer_state_dict"])
            if self._ema_on():
                if "ema_state_dict" in checkpoint:
                    self.optimizer.load_ema_state_dict(checkpoint["ema_state_dict"], checkpoint["ema_updates"])
                else:
                    self.optimizer.reset_ema()
                    print("Info: the checkpoint has no weight EMA; the EMA starts from the loaded weights")
            if scheduler is not None:
                scheduler.lambda_lr.load_state_dict(checkpoint["scheduler_state_dict"])
            epoch = checkpoint["epoch"]
            best_loss = checkpoint["best_loss"]
            if ("val_loss" in checkpoint) != (self.validation is not None):
                # a training loss and a held-out loss are not comparable: the best checkpoint is chosen afresh
                print(f"Info: the checkpoint's best loss is a {'validation' if 'val_loss' in checkpoint else 'training'} "
                      f"loss but this run selects by {'validation' if self.validation is not None else 'training'} "
                      "loss; the best loss restarts at inf")
                best_loss = float("inf")
            print(f"Resumed from ({checkpoint_path}) epoch {epoch}, best loss {best_loss:.6f}")
        else:
            print(f"No checkpoint ({checkpoint_path}) found. Starting from scratch.")
            epoch = 0
            best_loss = float("inf")
        return epoch, best_loss, scheduler

    def save_checkpoint(self, scheduler, epoch, best_loss, checkpoint_path, **extra):
        """Writes the reference's checkpoint dictionary; `extra` keys (validation: `val_loss`) are added to it."""
        if self._ema_on() and self.optimizer._ema_swapped:
            # the network holds the EMA: model_state_dict would lose the live weights
            raise RuntimeError("save_checkpoint() inside ema_weights()")
        sd = {k: v.detach().contiguous().cpu() for k, v in self.model.state_dict().items()}
        ck = {
            "epoch": epoch,
            "model_state_dict": sd,
            "optimizer_state_dict": self.optimizer.state_dict(),
            "scheduler_state_dict": (scheduler.lambda_lr.state_dict() if scheduler is not None else None),
            "best_loss": best_loss,
        }
        if self._ema_on():   # the EMA in the model's state-dict format: UNet1d.load_state_dict takes it as it is
            ck["ema_state_dict"] = self.optimizer.ema_state_dict(device="cpu")
            ck["ema_updates"] = self.optimizer.ema_updates
        ck.update(extra)
        torch.save(ck, checkpoint_path)

    def _ema_on(self):
        return isinstance(self.optimizer, FusedAdamW) and self.optimizer.ema_decay is not None

    @contextlib.contextmanager
    def ema_weights(self):
        """Inside the context the network holds the EMA of its weights (`ema_decay`), so `sample`, `sample_windows`,
        `predict_batch`, `predict_windows` and direct forward calls use it; the live weights are back, bit for bit, on
        exit.  Under data parallelism every rank must enter it (the sharded EMA is all-gathered)."""
        if not self._ema_on():
            raise RuntimeError("no weight EMA: set ema_decay before the optimizer is created (training starts)")
        self.optimizer.swap_ema()
        try:
            yield self.model
        finally:
            self.optimizer.swap_ema()

    def predict(self, dataloader, mixture_weights=(0.5, 0.5), num_steps=1000):
        self.model.eval()
        preds = np.array([])
        for ms2_1, ms1_1, ms2_2, ms1_2 in dataloader:
            x_0, ms1_cond, ms2_cond = self._mix_to_device(ms2_1, ms1_1, ms2_2, mixture_weights)
            pred, _ = self._predict_one_batch(x_0, ms2_cond=ms2_cond, ms1_cond=ms1_cond, num_steps=num_steps)
            preds = np.append(preds, {
                "ms2_1": ms2_1.cpu().detach().numpy(),
                "ms1_1": ms1_1.cpu().detach().numpy(),
                "mixture": ms2_cond.cpu().detach().numpy(),
                "pred": pred,
            })
        return preds

    def log_single_prediction(self, *args, **kwargs):
        try:
            import pyopenms_viz  # noqa: F401
        except ImportError:
            raise ImportError("pyopenms_viz is required for plotting predictions (as in the reference); "
                              "plotting is outside the B200 hot path")
        raise NotImplementedError("plotting / wandb prediction tables are out of scope of the B200 build")

    plot_single_prediction = log_single_prediction

    # ---------------------------------------------------------------------------------------- private
    def _init_for_training(self):
        self.loss_func = torch.nn.L1Loss()

    def _prepare_training(self, lr: float, **kwargs):
        self.model.train()
        self._set_lr(lr)

    def _set_optimizer(self, lr):
        if hasattr(self.model, "flat_params"):
            self.optimizer = FusedAdamW(self.model, lr=lr, ema_decay=self.ema_decay)
            plan = self._shard_plan()
            if plan:
                self.optimizer.set_sharding(torch.distributed.get_rank(), torch.distributed.get_world_size(), plan)
        else:  # an arbitrary user module (not the B200 denoiser): plain torch AdamW as in the reference
            if self.ema_decay is not None:
                raise ValueError("ema_decay needs a model with the flat-buffer API (the B200 UNet1d)")
            self.optimizer = torch.optim.AdamW(self.model.parameters(), lr=lr)

    def _set_lr(self, lr: float):
        if self.optimizer is None:
            self._set_optimizer(lr)
        else:
            for g in self.optimizer.param_groups:
                g["lr"] = lr

    def _get_lr_schedule_with_warmup(self, warmup_epoch, epoch):
        if warmup_epoch > epoch:
            warmup_epoch = epoch // 2
        return self.lr_scheduler_class(self.optimizer, num_warmup_steps=warmup_epoch, num_training_steps=epoch)

    def _mix_to_device(self, ms2_1, ms1_1, ms2_2, mixture_weights):
        """x_0 = ms2_1, ms1_cond = ms1_1, ms2_cond = w0*ms2_1 + w1*ms2_2 (reference 1071-1075), mixed on the GPU."""
        dev = self.device
        x_0 = ms2_1.to(dev, non_blocking=True).float().contiguous()
        ms1_cond = ms1_1.to(dev, non_blocking=True).float().contiguous()
        other = ms2_2.to(dev, non_blocking=True).float().contiguous()
        if x_0.is_cuda:
            ms2_cond = torch.empty_like(x_0)
            N.call("dq_mix_affine", x_0, other, float(mixture_weights[0]), float(mixture_weights[1]), 1.0, 0.0,
                   ms2_cond, x_0.numel())
        else:
            ms2_cond = x_0 * mixture_weights[0] + other * mixture_weights[1]
        return x_0, ms1_cond, ms2_cond

    def _train_one_epoch(self, epoch, dataloader, mixture_weights=(0.5, 0.5)):
        self.model.train()
        batch_loss = []
        for batch_idx, (ms2_1, ms1_1, ms2_2, ms1_2) in enumerate(dataloader):
            x_0, ms1_cond, ms2_cond = self._mix_to_device(ms2_1, ms1_1, ms2_2, mixture_weights)
            loss = self._train_one_batch(x_0, ms2_cond=ms2_cond, ms1_cond=ms1_cond, noise=None,
                                         ms1_loss_weight=self.ms1_loss_weight)
            batch_loss.append(loss)
            if self.use_wandb and self._is_rank0():
                import wandb
                wandb.log({"batch/train_loss": loss, "batch": batch_idx + epoch * len(dataloader)})
        return batch_loss

    def _dist_on(self):
        dist = torch.distributed
        return dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1

    def _shard_plan(self):
        """Flat ranges that are reduce-scattered and updated by one rank each (the four 300 M-parameter mid-block
        convolutions and the mid attention projections: 99 % of the parameters), or None: plain all-reduce and a
        replicated optimizer (one GPU, non-NCCL backends, DQ_SHARDED_OPT=0, modules without the flat-buffer API)."""
        if hasattr(self, "_shard_plan_cache"):
            return self._shard_plan_cache
        plan = None
        dist = torch.distributed
        if (self._dist_on() and os.environ.get("DQ_SHARDED_OPT", "1") != "0" and hasattr(self.model, "early_grad_ranges")
                and dist.get_backend() == "nccl"):
            ws = dist.get_world_size()
            plan = sorted((int(o), int(n)) for o, n in self.model.early_grad_ranges() if n % ws == 0 and n >= 1024 * ws) or None
        self._shard_plan_cache = plan
        return plan

    def _reduce_range(self, g, o, n, works):
        """Sum the gradient range [o, o + n) over the ranks: reduce-scatter (this rank keeps piece `rank`) if the range is
        in the shard plan, else an all-reduce in buckets."""
        dist = torch.distributed
        plan = self._shard_plan()
        if plan and (o, n) in plan:
            ws, rank = dist.get_world_size(), dist.get_rank()
            k = n // ws
            works.append(dist.reduce_scatter_tensor(g[o + rank * k:o + (rank + 1) * k], g[o:o + n], op=dist.ReduceOp.SUM,
                                                    async_op=True))
            return
        for s in range(o, o + n, self.grad_bucket_elems):
            e = min(o + n, s + self.grad_bucket_elems)
            works.append(dist.all_reduce(g[s:e], op=dist.ReduceOp.SUM, async_op=True))

    def _early_allreduce(self, ranges):
        """Called from the denoiser's backward as soon as the mid-stage gradients are final: start their
        reduction (async, NCCL stream) so it overlaps the down-path backward."""
        g = self.model.flat_grads()
        self._early_reduced = list(getattr(self, "_early_reduced", []))
        self._early_works = list(getattr(self, "_early_works", []))
        for (o, n) in ranges:
            self._reduce_range(g, int(o), int(n), self._early_works)
            self._early_reduced.append((int(o), int(n)))

    def _allreduce_grads(self):
        """Sum the flat gradient over the ranks (NCCL over NVLink; gloo in the CPU tests).  Returns the factor that
        turns the sum into the mean: with the fused optimizer it is folded into the clip coefficient (no pass over the
        gradient), otherwise the gradient is scaled here and 1.0 is returned."""
        dist = torch.distributed
        if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
            return 1.0
        ws = dist.get_world_size()
        if hasattr(self.model, "flat_grads"):
            g = self.model.flat_grads()[: self.model.n_trainable_flat]
            done = getattr(self, "_early_reduced", [])
            works = []
            todo = [r for r in (self._shard_plan() or []) if r not in done]   # sharded ranges nobody reduced early
            covered = sorted(list(done) + todo)
            pos = 0
            for (o, n) in covered:
                if o > pos:
                    self._reduce_range(g, pos, o - pos, works)
                pos = o + n
            if pos < g.numel():
                self._reduce_range(g, pos, g.numel() - pos, works)
            for (o, n) in todo:
                self._reduce_range(g, o, n, works)
            for w in getattr(self, "_early_works", []) + works:
                w.wait()
            self._early_reduced, self._early_works = [], []
            if isinstance(self.optimizer, FusedAdamW):
                return 1.0 / ws
            g.mul_(1.0 / ws)
            return 1.0
        for p in self.model.parameters():
            if p.grad is not None:
                dist.all_reduce(p.grad)
                p.grad.mul_(1.0 / ws)
        return 1.0

    def _auto_micro_batch(self, x_0):
        """Samples per forward/backward pass when `micro_batch` is not set: the whole batch if its saved activations
        fit, else as many samples as fit in 60 % of the free HBM (measured: ~1.1 kB of saved activations per
        (rt, mz) element of one sample for the default U-Net depth; 112 GB peak at 64 samples of 34 x 40000)."""
        b = x_0.shape[0]
        if not (x_0.is_cuda and x_0.dim() == 3):
            return b
        free, _ = torch.cuda.mem_get_info(x_0.device)
        # blocks cached by torch's allocator are reusable: count them as free
        free += torch.cuda.memory_reserved(x_0.device) - torch.cuda.memory_allocated(x_0.device)
        per_sample = 1100.0 * x_0.shape[1] * x_0.shape[2]
        return max(1, min(b, 64, int(0.6 * free / per_sample)))

    def _train_one_batch(self, x_0, ms2_cond=None, ms1_cond=None, noise=None, ms1_loss_weight=0.0, t=None):
        self.optimizer.zero_grad()
        if hasattr(self.model, "grad_ready_callback"):
            self.model.grad_ready_callback = self._early_allreduce if self._dist_on() else None
        b = x_0.shape[0]
        if self.micro_batch:
            mb = min(int(self.micro_batch), b)
        else:
            mb = self._auto_micro_batch(x_0)
        total = None
        n_mb = (b + mb - 1) // mb
        for k, s in enumerate(range(0, b, mb)):
            sl = slice(s, min(b, s + mb))
            w = (sl.stop - sl.start) / b
            kw = {} if t is None else {"t": t[sl]}
            if hasattr(self.model, "_final_microbatch"):
                self.model._final_microbatch = (k == n_mb - 1)
            if hasattr(self.model, "_wgrad_defer") and n_mb > 1 and x_0.dim() == 3:
                # mid-stage weight gradients: one GEMM per optimizer step over the K-concatenated micro-batches
                rp = x_0.shape[1] + 2
                self.model._wgrad_defer = (s * rp, b * rp, k == n_mb - 1)
            loss = self.train_step(
                x_0[sl],
                ms2_cond=None if ms2_cond is None else ms2_cond[sl],
                ms1_cond=None if ms1_cond is None else ms1_cond[sl],
                noise=None if noise is None else noise[sl],
                ms1_loss_weight=ms1_loss_weight or 0.0,
                **kw,
            )
            lm = loss.mean() * w
            lm.backward()
            total = lm.detach() if total is None else total + lm.detach()
        if hasattr(self.model, "_wgrad_defer"):
            self.model._wgrad_defer = None
        gscale = self._allreduce_grads()
        if isinstance(self.optimizer, FusedAdamW):
            self.optimizer.step(max_grad_norm=self.max_grad_norm, grad_scale=gscale, defer_gather=True)
        else:
            torch.nn.utils.clip_grad_norm_(self.model.parameters(), max_norm=self.max_grad_norm)
            self.optimizer.step()
        self.last_loss = total
        return total.item()

    def _predict_one_batch(self, x_0, ms2_cond=None, ms1_cond=None, num_steps=1000):
        self.model.eval()
        with torch.no_grad():
            sample, pred_noise = self.sample(torch.randn_like(x_0), ms2_cond=ms2_cond, ms1_cond=ms1_cond,
                                             num_steps=num_steps)
        return sample[0].cpu().detach().numpy(), pred_noise[0].cpu().detach().numpy()

    def predict_batch(self, x_T, ms2_cond, ms1_cond, num_steps=50, target=None, sampler="reference"):
        """Batched multi-window prediction that keeps EVERY window (the reference's `_predict_one_batch` returns item
        [0] only, model_interface.py:1150).  With `target` (the clean maps, values in [0, 1]) it also returns the cheap
        evaluation metric of SURVEY.md §8f-2: the per-window cosine similarity between prediction and target, from one
        fused pass (dq_cosine_sums).  `sampler` is passed to `sample`.  Returns (pred, pred_noise) or (pred, pred_noise,
        cosine (b,))."""
        self.model.eval()
        with torch.no_grad():
            pred, pred_noise = self.sample(x_T, ms2_cond=ms2_cond, ms1_cond=ms1_cond, num_steps=num_steps,
                                           sampler=sampler)
            if target is None:
                return pred, pred_noise
            return pred, pred_noise, self.cosine_to_target(pred, target)

    @staticmethod
    def cosine_to_target(pred, target):
        """Per-window cosine similarity <p, t> / (|p| |t|) of (b, rt, mz) maps, one kernel."""
        b = pred.shape[0]
        sums = torch.zeros(b, 3, dtype=torch.float32, device=pred.device)
        N.call("dq_cosine_sums", pred.float().contiguous(), target.to(pred.device).float().contiguous(), sums,
               pred.numel() // b, b)
        return sums[:, 0] / (sums[:, 1].sqrt() * sums[:, 2].sqrt()).clamp_min(1e-30)

    @staticmethod
    def map_scores(pred, truth):
        """The 9 float64 sums of `dq_map_scores` per window of (b, rt, mz) maps, one deterministic pass: sse, <p, g>,
        |p|^2, |g|^2, the same three of the RT-summed spectra, and the weighted XIC correlation sums.  Turn them into
        scores with `dquartic.utils.validation.finalize_scores`.  Returns (b, 9) float64 on the maps' device."""
        if pred.dim() != 3 or tuple(pred.shape) != tuple(truth.shape):
            raise ValueError(f"map_scores needs two (b, rt, mz) maps of one shape, got {tuple(pred.shape)} and "
                             f"{tuple(truth.shape)}")
        b, rt, mz = pred.shape
        pred = pred.float().contiguous()
        truth = truth.to(pred.device).float().contiguous()
        part = torch.empty(b * N.map_scores_nblk(mz) * 9, dtype=torch.float64, device=pred.device)
        out = torch.empty(b, 9, dtype=torch.float64, device=pred.device)
        N.call("dq_map_scores", pred, truth, part, out, b, rt, mz)
        return out

    def _gather_windows(self, local, n_windows, rank, world):
        """Per-window rows (n_local, k) of this rank's `shard_windows` block -> all (n_windows, k) rows in window order on
        every rank (padded all-gather) when a process group is up; otherwise the local block as it is."""
        dist = torch.distributed
        if not (dist.is_available() and dist.is_initialized()) or world == 1:
            return local
        width = -(-n_windows // world)
        buf = torch.zeros(width, local.shape[1], dtype=local.dtype, device=self.device)
        buf[:local.shape[0]].copy_(local)
        out = torch.empty(world * width, local.shape[1], dtype=local.dtype, device=self.device)
        dist.all_gather_into_tensor(out, buf)
        blocks = []
        for r in range(world):
            lo, hi = self.shard_windows(n_windows, r, world)
            blocks.append(out[r * width:r * width + hi - lo])
        return torch.cat(blocks)

    def _rank_world(self, rank, world):
        if rank is None or world is None:
            dist = torch.distributed
            on = dist.is_available() and dist.is_initialized()
            return (dist.get_rank(), dist.get_world_size()) if on else (0, 1)
        return int(rank), int(world)

    def validate(self, vset, chunk=64, rank=None, world=None):
        """Held-out denoising loss of the current weights on `vset` (a `ValidationSet`): the per-sample loss of
        `denoising_loss` for every (window, band) row at the band's timestep t_k and the window's fixed noise, `chunk`
        rows per forward.  Windows are split by `shard_windows(W, rank, world)` (default: torch.distributed's rank and
        world size); under a process group the per-window losses are all-gathered and every rank reduces them in window
        order, otherwise the local block is returned.  Returns {"bands", "loss_by_band" (K,), "val_loss", "per_window"
        (n, K), "windows" (lo, hi)}, float64 numpy; val_loss = mean_k loss_weight[t_k] loss_by_band[k], the training
        objective (without the SIC term) under stratified t."""
        rank, world = self._rank_world(rank, world)
        W, bands = vset.windows, list(vset.bands)
        K = len(bands)
        lo, hi = self.shard_windows(W, rank, world)
        rows = [(w, k) for w in range(lo, hi) for k in range(K)]
        local = torch.zeros(hi - lo, K, dtype=torch.float64, device=self.device)
        was_training = self.model.training
        self.model.eval()
        try:
            for s in range(0, len(rows), int(chunk)):
                rr = rows[s:s + int(chunk)]
                wi = torch.tensor([w for w, _ in rr], device=self.device)
                t = torch.tensor([bands[k] for _, k in rr], device=self.device)
                loss = self.denoising_loss(vset.x0[wi], vset.cond[wi], vset.m1[wi], t, vset.noise[wi])
                local.view(-1)[s:s + len(rr)] = loss
        finally:
            self.model.train(was_training)
        per = self._gather_windows(local, W, rank, world).cpu().numpy()
        by_band = per.mean(axis=0)
        lw = self.loss_weight.detach().double().cpu().numpy()[bands]
        return {"bands": bands, "loss_by_band": by_band, "val_loss": float(np.mean(lw * by_band)), "per_window": per,
                "windows": (0, W) if per.shape[0] == W else (lo, hi)}

    def score_samples(self, vset, sampler="dpm++2m", num_steps=20, seed=0, chunk=32, rank=None, world=None):
        """Sample the validation mixtures of `vset` through `sample_windows` (window id = mixture index, x_T from
        (seed, id)) and score every map against its clean map with `dq_map_scores`.  Sharding and gather as `validate`.
        Returns {"per_window": {cosine, rmse, spectral_angle, xic_corr: (n,) arrays}, "mean": {the same: floats},
        "windows": (lo, hi)}."""
        from ..utils.validation import SCORE_KEYS, finalize_scores

        rank, world = self._rank_world(rank, world)
        W = vset.windows
        lo, hi = self.shard_windows(W, rank, world)

        def cond_fn(ids):
            idx = torch.tensor(ids, device=self.device)
            return vset.cond[idx], vset.m1[idx]

        _, maps = self.sample_windows(range(W), cond_fn, seed=seed, num_steps=num_steps, chunk=chunk, rank=rank,
                                      world=world, sampler=sampler)
        local = torch.zeros(hi - lo, 9, dtype=torch.float64, device=self.device)
        for s in range(0, hi - lo, int(chunk)):
            e = min(hi - lo, s + int(chunk))
            local[s:e] = self.map_scores(maps[s:e].to(self.device), vset.x0[lo + s:lo + e])
        sums = self._gather_windows(local, W, rank, world)
        sc = finalize_scores(sums, vset.x0.shape[1], vset.x0.shape[2])
        per = {k: sc[k] for k in SCORE_KEYS}
        return {"per_window": per, "mean": {k: float(np.mean(v)) for k, v in per.items()},
                "windows": (0, W) if sums.shape[0] == W else (lo, hi)}

    def predict_windows(self, dataloader, mixture_weights=(0.5, 0.5), num_steps=50, seed=0, sampler="reference"):
        """`predict` for throughput: every batch item is kept and scored.  Returns a list of dicts
        {ms2_1, ms1_1, mixture, pred, cosine} per batch (numpy arrays; `cosine` is pred vs ms2_1 per window)."""
        out = []
        g = torch.Generator(device=self.device)
        g.manual_seed(int(seed))
        for ms2_1, ms1_1, ms2_2, ms1_2 in dataloader:
            x_0, ms1_cond, ms2_cond = self._mix_to_device(ms2_1, ms1_1, ms2_2, mixture_weights)
            x_T = torch.empty_like(x_0).normal_(generator=g)
            pred, _, cos = self.predict_batch(x_T, ms2_cond, ms1_cond, num_steps=num_steps, target=x_0,
                                              sampler=sampler)
            out.append({"ms2_1": x_0.cpu().numpy(), "ms1_1": ms1_cond.cpu().numpy(), "mixture": ms2_cond.cpu().numpy(),
                        "pred": pred.cpu().numpy(), "cosine": cos.cpu().numpy()})
        return out
