"""Host-side mirrors of the reference training drivers for the hot path.

`rollout_train` restates `Trainer.rollout_model` (trainer/trainer.py:144-159: whole batch, fixed step) and
`R_Trainer.rollout_model` (trainer/r_trainer.py:112-133: per-sample B=1 while-loops with out_T=1.5, window NOT
detached => BPTT through the chained model calls) around the drop-in module; `train_step` is the body of
`train_one_epoch` (trainer.py:178-198 / r_trainer.py:145-159): rollout -> MSE(+rt penalty) -> backward -> clip ->
optimizer step.  All model arithmetic (forward AND backward) runs in libtante_b200.so; loss, clipping and the
optimizer are the reference's own torch calls (optim is out of scope, SURVEY.md §2), and data-parallel training adds
exactly one collective: an all-reduce of ONE flat gradient bucket before clipping (SURVEY.md §8(e)).
"""
from __future__ import annotations

from typing import Optional

import math
import os

import torch
import torch.distributed as dist


def mse_loss(y_pred, y_ref, rts=None, eps: float = 0.5, n: int = 2):
    """trainer/metrics.py:19-80: MSE.eval (mean over H, W) .mean() [+ MSE.eval_rt penalty on mean R_t]."""
    loss = torch.mean((y_pred - y_ref) ** 2, dim=(-3, -2)).mean()
    if rts is None:
        return loss
    avg = torch.mean(rts)
    up, down = min(1 + eps, 4), max(1 + eps, 4)
    a = float(avg)                                   # the reference's Python `if` on a tensor: a host sync
    if a < up:
        loss = loss + 5e-3 * (up - avg) ** n
    if a > down:
        loss = loss + 1e-1 * (avg - down) ** n
    return loss


class _FusedMSE(torch.autograd.Function):
    """mean((y_pred - y_ref)^2) over every element -- what `MSE.eval(...).mean()` (trainer/metrics.py:53-80) computes
    on the concatenated, channels-last predictions -- evaluated directly on the per-call channels-first frame tensors
    by libtante_b200's `tante_mse_cl`: one pass for the loss, one for the gradients; no permute / cat / sub / pow / mean
    kernels and none of their autograd counterparts."""

    @staticmethod
    def forward(ctx, y_ref, n_steps, *frames):
        from . import _abi
        lib = _abi.load()
        dev = frames[0].device
        y_ref = y_ref.to(torch.float32).contiguous()
        B, n_ref, H, W, D = y_ref.shape
        stream = torch.cuda.current_stream(dev).cuda_stream
        acc = torch.zeros(1, device=dev, dtype=torch.float32)
        plan, f0 = [], 0
        for f in frames:
            if f.dtype != torch.float32 or not f.is_contiguous() or f.shape[0] != B or tuple(f.shape[2:]) != (D, H, W):
                raise ValueError("fused MSE expects contiguous fp32 frames (B, n, D, H, W) matching y_ref (B, n, H, W, D)")
            use = max(0, min(int(f.shape[1]), n_steps - f0))
            plan.append((f0, use))
            if use > 0:
                _abi.check(lib.tante_mse_cl(f.data_ptr(), y_ref.data_ptr(), B, int(f.shape[1]), use, D, H * W, n_ref, f0,
                                            0.0, None, acc.data_ptr(), None, stream))
            f0 += use
        ctx.numel = float(B) * n_steps * H * W * D
        ctx.plan, ctx.n_ref = plan, n_ref
        ctx.save_for_backward(y_ref, *frames)
        return (acc / ctx.numel).reshape(())

    @staticmethod
    def backward(ctx, gout):
        from . import _abi
        lib = _abi.load()
        y_ref, *frames = ctx.saved_tensors
        B, n_ref, H, W, D = y_ref.shape
        dev = y_ref.device
        stream = torch.cuda.current_stream(dev).cuda_stream
        g = gout.to(torch.float32).contiguous()
        grads = []
        for f, (f0, use) in zip(frames, ctx.plan):
            gf = torch.empty_like(f)
            _abi.check(lib.tante_mse_cl(f.data_ptr(), y_ref.data_ptr(), B, int(f.shape[1]), use, D, H * W, n_ref, f0,
                                        2.0 / ctx.numel, g.data_ptr(), None, gf.data_ptr(), stream))
            grads.append(gf)
        return (None, None, *grads)


def mse_loss_frames(frames, y_ref, n_steps: int):
    """MSE.eval(...).mean() on the per-call channels-first predictions (list of (B, n_i, D, H, W)) against the
    channels-last targets y_ref (B, >= n_steps, H, W, D); frames beyond n_steps are ignored (r_trainer.py:130)."""
    return _FusedMSE.apply(y_ref, int(n_steps), *frames)


def _bptt_windows(model, window) -> bool:
    """The module's one-node BPTT rollout (TANTE.rollout_train) applies: CUDA input, the windowed entry points cover the
    configuration, grad mode, and TANTE_BPTT_WINDOWS is not 0."""
    return (hasattr(model, "rollout_train") and window.is_cuda and getattr(model, "bptt_windows_ok", True)
            and torch.is_grad_enabled() and os.environ.get("TANTE_BPTT_WINDOWS", "1") != "0")


def _roll_frames(model, window, n_steps: int):
    """`_roll` for the fixed-step model without the formatter permute and the cat over calls."""
    if int(getattr(model, "output_length", 0)) == 1 and _bptt_windows(model, window):
        return [model.rollout_train(window, n_steps)]      # one autograd node, the window slides over one history buffer
    moving, ys, cum = window, [], 0
    while cum < n_steps:
        y = model(moving)
        cum += y.shape[1]
        if cum < n_steps:
            moving = torch.cat([moving[:, y.shape[1]:], y], dim=1)      # window NOT detached (BPTT)
        ys.append(y)
    return ys


def _roll(model, window, n_steps: int, out_T):
    moving, ys, rts, cum = window, [], [], 0
    while cum < n_steps:
        if model.deg:
            y, rt = model(moving), None
        else:
            y, rt = model(moving, out_T)
        cum += y.shape[1]
        if cum < n_steps:
            moving = torch.cat([moving[:, y.shape[1]:], y], dim=1)      # window NOT detached (r_trainer.py:126)
        ys.append(y.permute(0, 1, 3, 4, 2))                             # formatter.process_output
        if rt is not None:
            rts.append(rt)
    return torch.cat(ys, dim=1)[:, :n_steps], (torch.cat(rts, dim=0) if rts else None)


def flat_rts(rts, ns, every_call: bool = False):
    """Per-call R_t (n_calls, B) and frames per call (n_calls, B) of the batched adaptive rollout -> the flat Rts of the
    per-sample loops (r_trainer.py:118-131): sample 0's calls in order, then sample 1's, ...; entries of calls a sample did
    not take part in (ns == 0) are left out.  every_call: every sample took part in every call (no mask, no host sync)."""
    rt = rts.t()
    return rt.reshape(-1) if every_call else rt[ns.t() > 0]


def rollout_train(model, x, n_steps: int, out_T: float = 1.5):
    """x (B,T,D,H,W) channels-first -> (y_pred (B,n_steps,H,W,D), Rts or None)."""
    if model.deg:
        return _roll(model, x, n_steps, out_T)
    if _bptt_windows(model, x):
        # the per-sample loops below as one batched device-resident rollout (TANTE.rollout_train, deg=False)
        pred, rts, ns, _ = model.rollout_train(x, n_steps, out_T=out_T)
        return pred.permute(0, 1, 3, 4, 2), flat_rts(rts, ns, every_call=int(math.floor(out_T + 0.001)) <= 1)
    outs, rts = [], []
    for b in range(x.shape[0]):                                         # r_trainer.py:118 ("TODO: batch size > 1")
        y, r = _roll(model, x[b:b + 1], n_steps, out_T)
        outs.append(y)
        rts.append(r)
    return torch.cat(outs, dim=0), torch.cat(rts, dim=0)


class GradBucket:
    """One flat fp32 gradient bucket: every `p.grad` is a view into it, so autograd accumulates in place and
    data-parallel training needs a single all-reduce (NCCL over NVLink) per optimizer step."""

    def __init__(self, model: torch.nn.Module):
        self.params = [p for p in model.parameters() if p.requires_grad]
        dev = self.params[0].device
        named = dict(model.named_parameters())
        if hasattr(model, "grad_layout") and dev.type == "cuda" and all(p.requires_grad for p in named.values()):
            # the library's own flat layout: the backward then accumulates with ONE add per model call
            names, offsets, n = model.grad_layout(dev)
            self.flat = torch.zeros(n, device=dev, dtype=torch.float32)
            for name, off in zip(names, offsets):
                p = named[name]
                if p.dtype == torch.complex64:      # SpectralLayer.weight: (re, im) float pairs in the flat buffer
                    p.grad = torch.view_as_complex(self.flat[off:off + 2 * p.numel()].view(*p.shape, 2))
                else:
                    p.grad = self.flat[off:off + p.numel()].view_as(p)
            return
        n = sum(p.numel() for p in self.params)
        self.flat = torch.zeros(n, device=dev, dtype=torch.float32)
        off = 0
        for p in self.params:
            p.grad = self.flat[off:off + p.numel()].view_as(p)
            off += p.numel()

    def zero(self):
        self.flat.zero_()

    def all_reduce_mean(self):
        if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
            dist.all_reduce(self.flat, op=dist.ReduceOp.SUM)
            self.flat.mul_(1.0 / dist.get_world_size())

    # ---- native data-parallel exchange (tante_allreduce_grads: SURVEY.md 8(b) / 8(e)) ----------------------------------
    def init_native_comm(self, model) -> bool:
        """One NCCL communicator inside the library (tante_comm_init), its id broadcast through torch.distributed.
        Returns False (and changes nothing) outside a multi-rank CUDA job or when TANTE_NATIVE_ALLREDUCE=0."""
        import os
        self._native = None
        if not (dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1 and self.flat.is_cuda):
            return False
        if os.environ.get("TANTE_NATIVE_ALLREDUCE", "1") == "0" or not hasattr(model, "grad_layout"):
            return False
        import ctypes
        from . import _abi
        eng = model._engine(self.flat.device)
        buf = ctypes.create_string_buffer(128)
        if dist.get_rank() == 0:
            _abi.check(eng.lib.tante_comm_unique_id(buf))
        box = [bytes(buf.raw)]
        dist.broadcast_object_list(box, src=0)
        _abi.check(eng.lib.tante_comm_init(eng.handle, box[0], dist.get_world_size(), dist.get_rank()))
        self._native = eng
        return True

    def all_reduce_sum(self) -> int:
        """SUM all-reduce of the flat bucket on the current stream; returns the world size (the 1 / world scaling is folded
        into the optimizer step).  Uses the library's communicator when init_native_comm succeeded."""
        if not (dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1):
            return 1
        eng = getattr(self, "_native", None)
        if eng is not None:
            from . import _abi
            stream = torch.cuda.current_stream(self.flat.device).cuda_stream
            _abi.check(eng.lib.tante_allreduce_grads(eng.handle, self.flat.data_ptr(), None, stream))
        else:
            dist.all_reduce(self.flat, op=dist.ReduceOp.SUM)
        return dist.get_world_size()


def train_step(model, optimizer, x, y_ref, n_steps: int = 4, bucket: Optional[GradBucket] = None,
               clip: str = "norm", rt_eps: float = 0.5, rt_n: int = 2):
    """One optimizer step.  clip = "norm": clip_grad_norm_(1.0) (trainer.py:192-193); "value": clip_grad_value_(1.0)
    (r_trainer.py:155).  Returns the (device) loss tensor."""
    if getattr(model, "deg", False) and x.is_cuda and hasattr(model, "grad_layout"):
        # fixed-step model on the CUDA path: loss and its gradient straight from the per-call frames (tante_mse_cl)
        loss = mse_loss_frames(_roll_frames(model, x, n_steps), y_ref, n_steps)
    else:
        y_pred, rts = rollout_train(model, x, n_steps)
        loss = mse_loss(y_pred, y_ref, rts, rt_eps, rt_n)
    if bucket is not None:
        bucket.zero()
    else:
        optimizer.zero_grad(set_to_none=True)
    loss.backward()
    from .optim import FusedAdamW
    if isinstance(optimizer, FusedAdamW) and bucket is not None:
        # all-reduce (sum) + mean + clip + AdamW + repack: the NCCL kernel and three launches of the library
        world = bucket.all_reduce_sum()
        optimizer.step(clip=clip, clip_value=1.0, grad_scale=1.0 / world)
        return loss.detach()
    if bucket is not None:
        bucket.all_reduce_mean()          # before clipping: clipping must see the averaged gradient
    params = bucket.params if bucket is not None else list(model.parameters())
    if clip == "norm":
        torch.nn.utils.clip_grad_norm_(params, 1.0)
    elif clip == "value":
        torch.nn.utils.clip_grad_value_(params, 1.0)
    optimizer.step()
    return loss.detach()


# =====================================================================================================
# Drop-ins for trainer.Trainer / trainer.R_Trainer (configs/tante.yaml:48 `trainer._target_`)
# =====================================================================================================
def _wandb_log(logs, step):
    """wandb.log if a run is active (train.py:68-76 opens it); silently nothing otherwise."""
    try:
        import wandb
        if getattr(wandb, "run", None) is not None:
            wandb.log(logs, step=step)
    except Exception:
        pass


class _TrainerBase:
    """Shared body of the two reference trainers: constructor kwargs, `save_model` / `load_checkpoint` (checkpoint keys
    incl. the reference's `optimizer_state_dit` spelling, trainer.py:112-137 / r_trainer.py:85-110), `train()` with
    `recent.pt` every epoch and `best.pt` on improvement (trainer.py:232-255 / r_trainer.py:208-230)."""

    adaptive = False

    def _init_common(self, kw):
        import logging
        import os
        from .rollout import DefaultChannelsFirstFormatter
        for k, v in kw.items():
            if k != "self" and not k.startswith("_"):
                setattr(self, k, v)
        self._log = logging.getLogger(__name__)
        self._os = os
        self.device = torch.device(self.device)
        self.starting_epoch = 1
        self.amp_type = torch.bfloat16 if self.amp_type == "bfloat16" else torch.float16
        self.grad_scaler = torch.GradScaler(self.device.type, enabled=self.enable_amp and self.amp_type != torch.bfloat16)
        self.best_val_loss = None
        self.starting_val_loss = float("inf")
        self.dset_metadata = getattr(getattr(self.datamodule, "train_dataset", None), "metadata", None)
        if self.formatter != "channels_first_default":
            raise NotImplementedError("only channels_first_default is wired to the CUDA model")
        self.formatter = DefaultChannelsFirstFormatter(self.dset_metadata)
        self._bucket = None
        if self.checkpoint_path and len(self.checkpoint_path) > 0:
            self.load_checkpoint(self.checkpoint_path)

    def save_model(self, epoch: int, validation_loss: float, output_path: str):
        torch.save({"epoch": epoch, "model_state_dict": self.model.state_dict(),
                    "optimizer_state_dit": self.optimizer.state_dict(), "validation_loss": validation_loss,
                    "best_validation_loss": self.best_val_loss}, output_path)

    def load_checkpoint(self, checkpoint_path: str):
        self._log.info(f"Loading checkpoint from {checkpoint_path}")
        checkpoint = torch.load(checkpoint_path, weights_only=False)
        if self.model is not None:
            self.model.load_state_dict(checkpoint["model_state_dict"])
        if self.optimizer is not None:
            self.optimizer.load_state_dict(checkpoint["optimizer_state_dit"])
        self.best_val_loss = checkpoint["best_validation_loss"]
        self.starting_val_loss = checkpoint["validation_loss"]
        self.starting_epoch = checkpoint["epoch"] + 1
        if self.lr_scheduler:
            for _ in range(self.starting_epoch - 1):
                self.lr_scheduler.step()

    def _grad_bucket(self):
        """Data-parallel runs (is_distributed + an initialised process group) all-reduce ONE flat gradient bucket."""
        if self._bucket is None and self.is_distributed and dist.is_available() and dist.is_initialized() \
                and dist.get_world_size() > 1:
            self._bucket = GradBucket(self.model)
        return self._bucket

    def train(self):
        train_dataloader = self.datamodule.train_dataloader()
        val_dataloader = self.datamodule.val_dataloader()
        val_loss = self.starting_val_loss
        join = self._os.path.join
        for epoch in range(self.starting_epoch, self.max_epoch + 1):
            if self.is_distributed and hasattr(getattr(train_dataloader, "sampler", None), "set_epoch"):
                train_dataloader.sampler.set_epoch(epoch)
            self._log.info(f"Epoch {epoch}/{self.max_epoch}: starting training")
            train_loss, train_logs = self.train_one_epoch(epoch, train_dataloader)
            self._log.info(f"Epoch {epoch}/{self.max_epoch}: avg training loss {train_loss}")
            _wandb_log(train_logs, epoch)
            self.save_model(epoch, val_loss, join(self.checkpoint_folder, "recent.pt"))
            self._log.info(f"Epoch {epoch}/{self.max_epoch}: starting validation")
            val_loss = self.validation_loop(val_dataloader, epoch=epoch)
            self._log.info(f"Epoch {epoch}/{self.max_epoch}: avg validation loss {val_loss}")
            _wandb_log({"valid": val_loss}, epoch)
            if self.best_val_loss is None or val_loss < self.best_val_loss:
                self.save_model(epoch, val_loss, join(self.checkpoint_folder, "best.pt"))
                self.best_val_loss = val_loss


class Trainer(_TrainerBase):
    """Drop-in for trainer.Trainer (trainer.py:72-255): fixed-step model, whole-batch rollout with BPTT,
    `clip_grad_norm_(1.0)`.  The CViT branch (trainer.py:161-172) belongs to another model."""

    def __init__(self, checkpoint_folder: str = "", formatter: str = "channels_first_default", model=None, datamodule=None,
                 optimizer=None, train_loss_fn=None, eval_loss_fn=None, max_epoch: int = 1, lr_scheduler=None,
                 device=torch.device("cuda"), is_distributed: bool = False, enable_amp: bool = False,
                 amp_type: str = "float16", checkpoint_path: str = "", n_steps_output: int = 1, n_steps_rollout: int = 8,
                 rt_eps: float = 0.5, rt_n: int = 2, cvit: bool = False, num_query_points: int = 1024):
        if cvit:
            raise NotImplementedError("cvit=True selects the CViT query-point rollout (trainer.py:161-172), not TANTE")
        self._init_common(dict(locals()))

    def rollout_model(self, model, batch, formatter, mode="train"):
        n_steps = self.n_steps_output if mode == "train" else self.n_steps_rollout
        moving_batch, y_ref = formatter.process_input(batch)
        moving_batch = moving_batch[0].to(self.device)
        if mode != "train" and not torch.is_grad_enabled() and hasattr(model, "rollout"):
            from .rollout import rollout_eval
            y, _, _, _ = rollout_eval(model, moving_batch, n_steps)       # device-resident loop
            return y, y_ref.to(self.device)
        y_pred_out, _ = _roll(model, moving_batch, n_steps, 1.5)
        return y_pred_out, y_ref.to(self.device)

    def _fused_mse(self) -> bool:
        return (type(self.train_loss_fn).__name__ == "MSE" and getattr(self.model, "deg", False)
                and hasattr(self.model, "grad_layout") and self.device.type == "cuda")

    def train_one_epoch(self, epoch: int, dataloader):
        import time
        self.model.train()
        epoch_loss, train_logs = 0.0, {}
        start_time = time.time()
        bucket = self._grad_bucket()
        for i, batch in enumerate(dataloader):
            t0 = time.time()
            with torch.autocast(self.device.type, enabled=self.enable_amp, dtype=self.amp_type):
                if self._fused_mse():
                    # MSE(...).mean() straight from the per-call channels-first frames (tante_mse_cl): no permute / cat
                    moving, y_ref = self.formatter.process_input(batch)
                    y_ref = y_ref.to(self.device)
                    frames = _roll_frames(self.model, moving[0].to(self.device), self.n_steps_output)
                    forward_time = time.time() - t0
                    loss = mse_loss_frames(frames, y_ref, self.n_steps_output)
                else:
                    y_pred, y_ref = self.rollout_model(self.model, batch, self.formatter, "train")
                    forward_time = time.time() - t0
                    assert y_ref.shape == y_pred.shape, \
                        f"Mismatching shapes between reference {y_ref.shape} and prediction {y_pred.shape}"
                    loss = self.train_loss_fn(y_pred, y_ref, None).mean()
            if bucket is not None:
                bucket.zero()
            self.grad_scaler.scale(loss).backward()
            if bucket is not None:
                bucket.all_reduce_mean()
            self.grad_scaler.unscale_(self.optimizer)
            torch.nn.utils.clip_grad_norm_(self.model.parameters(), max_norm=1.0)
            self.grad_scaler.step(self.optimizer)
            self.grad_scaler.update()
            if bucket is None:
                self.optimizer.zero_grad()
            epoch_loss += loss.item() / len(dataloader)
            print(f"Epoch {epoch}, Batch {i+1}/{len(dataloader)}: loss {loss.item()}, forward time {forward_time}")
        train_logs["time_per_train_iter"] = (time.time() - start_time) / len(dataloader)
        train_logs["train_loss"] = epoch_loss
        if self.lr_scheduler:
            self.lr_scheduler.step()
            train_logs["lr"] = self.lr_scheduler.get_last_lr()[-1]
        return epoch_loss, train_logs

    @torch.inference_mode()
    def validation_loop(self, dataloader, epoch: int = 0) -> float:
        self.model.eval()
        seq_loss = 0.0
        with torch.autocast(self.device.type, enabled=self.enable_amp, dtype=self.amp_type):
            for batch in dataloader:
                y_pred, y_ref = self.rollout_model(self.model, batch, self.formatter, "eval")
                assert y_ref.shape == y_pred.shape, \
                    f"Mismatching shapes between reference {y_ref.shape} and prediction {y_pred.shape}"
                seq_loss += self.eval_loss_fn(y_pred, y_ref, None).mean().item()
        validation_loss = seq_loss / len(dataloader)
        with open(self.checkpoint_folder + "/saved_loss.txt", "a") as f:
            f.write(str(validation_loss) + "\n")
        return validation_loss


def rt_analyse(rt):
    """r_trainer.py:35-41."""
    step = len(rt)
    return torch.mean(rt).item(), step, (torch.std(rt, unbiased=True).item() if step > 1 else 0)


class R_Trainer(_TrainerBase):
    """Drop-in for trainer.R_Trainer (r_trainer.py:43-231): adaptive model, per-sample B=1 rollouts with out_T = 1.5 and
    BPTT through the chained calls, MSE + rt penalty, `clip_grad_value_(1.0)`.  On the CUDA module the per-sample loops run
    as one batched rollout (`rollout_train`); `train_out_T` (default 1.5, the reference's) sets the out_T of training."""

    adaptive = True

    def __init__(self, checkpoint_folder: str = "", formatter: str = "channels_first_default", model=None, datamodule=None,
                 optimizer=None, train_loss_fn=None, eval_loss_fn=None, max_epoch: int = 1, lr_scheduler=None,
                 device=torch.device("cuda"), is_distributed: bool = False, enable_amp: bool = False,
                 amp_type: str = "float16", checkpoint_path: str = "", n_steps_output: int = 4, n_steps_rollout: int = 8,
                 rt_eps: float = 0.5, rt_n: int = 2, train_out_T: float = 1.5):
        # train_out_T: out_T of the training rollout (the reference always uses 1.5, r_trainer.py:117-133)
        self._init_common(dict(locals()))

    def rollout_model(self, model, batch, formatter, mode="train"):
        n_steps = self.n_steps_output if mode == "train" else self.n_steps_rollout
        batch, y_ref = formatter.process_input(batch)
        batch = batch[0].to(self.device)
        if mode != "train" and not torch.is_grad_enabled() and hasattr(model, "rollout"):
            # the per-sample B=1 loops of r_trainer.py:118-129 as ONE device-resident per-sample rollout
            from .rollout import rollout_eval
            y, Rts, _, _ = rollout_eval(model, batch, n_steps, out_T=1.5, per_sample=True)
            return y, y_ref.to(self.device), Rts
        y_pred_out, Rts = rollout_train(model, batch, n_steps, self.train_out_T)
        return y_pred_out, y_ref.to(self.device), Rts

    def train_one_epoch(self, epoch: int, dataloader):
        import time
        self.model.train()
        epoch_loss, train_logs = 0.0, {}
        start_time = time.time()
        rt_saved, rt_var_saved, steps = [], [], []
        bucket = self._grad_bucket()
        for i, batch in enumerate(dataloader):
            t0 = time.time()
            with torch.autocast(self.device.type, enabled=self.enable_amp, dtype=self.amp_type):
                y_pred, y_ref, Rts = self.rollout_model(self.model, batch, self.formatter, "train")
                forward_time = time.time() - t0
                assert y_ref.shape == y_pred.shape, \
                    f"Mismatching shapes between reference {y_ref.shape} and prediction {y_pred.shape}"
                loss = self.train_loss_fn(y_pred, y_ref, Rts, self.rt_eps, self.rt_n)
            rt_avg, step, var = rt_analyse(Rts)
            if bucket is not None:
                bucket.zero()
            self.grad_scaler.scale(loss).backward()
            if bucket is not None:
                bucket.all_reduce_mean()
            torch.nn.utils.clip_grad_value_(self.model.parameters(), 1.0)
            self.grad_scaler.step(self.optimizer)
            self.grad_scaler.update()
            if bucket is None:
                self.optimizer.zero_grad()
            epoch_loss += loss.item() / len(dataloader)
            print(f"Epoch {epoch}, Batch {i+1}/{len(dataloader)}: loss {loss.item()}, steps {step/4}, var {var}, "
                  f"rt {rt_avg}, forward time {forward_time}")
            rt_saved.append(rt_avg)
            rt_var_saved.append(var)
            steps.append(step / 4)
        train_logs["time_per_train_iter"] = (time.time() - start_time) / len(dataloader)
        train_logs["train_loss"] = epoch_loss
        train_logs["rt"] = sum(rt_saved) / len(rt_saved)
        train_logs["rt_var"] = sum(rt_var_saved) / len(rt_var_saved)
        train_logs["steps"] = sum(steps) / len(steps)
        if self.lr_scheduler:
            self.lr_scheduler.step()
            train_logs["lr"] = self.lr_scheduler.get_last_lr()[-1]
        return epoch_loss, train_logs

    @torch.inference_mode()
    def validation_loop(self, dataloader, epoch: int = 0) -> float:
        self.model.eval()
        rt_list, seq_loss = [], 0.0
        with torch.autocast(self.device.type, enabled=self.enable_amp, dtype=self.amp_type):
            for batch in dataloader:
                y_pred, y_ref, Rts = self.rollout_model(self.model, batch, self.formatter, "eval")
                assert y_ref.shape == y_pred.shape, \
                    f"Mismatching shapes between reference {y_ref.shape} and prediction {y_pred.shape}"
                seq_loss += self.eval_loss_fn(y_pred, y_ref, None).mean().item()
                rt_list += Rts.tolist()
        validation_loss = seq_loss / len(dataloader)
        with open(self.checkpoint_folder + "/saved_loss.txt", "a") as f:
            f.write(str(validation_loss) + "\n")
        RT = sum(rt_list) / len(rt_list)
        with open(self.checkpoint_folder + "/saved_rt.txt", "a") as f:
            f.write(str(RT) + "\n")
        return validation_loss
