"""Training step around the hot path, mirroring gato/training/trainer.py:127-188 and schedulers.py:21-32.

What is reproduced exactly: the per-task batch split from the *_prop flags incl. the multinomial remainder draw
(trainer.py:134-154), forward/backward on the combined dict list, global-norm clip 1.0, AdamW(0.9/0.95, 1e-8, wd 0.1
on every parameter), linear warm-up + cosine decay, gradient accumulation.  The optimiser runs as one fused kernel
over the flat arenas (csrc/optim.cu); data parallelism is neko_b200.dp.  Evaluation / W&B / checkpoints are host
plumbing outside the hot path (utils.save_checkpoint writes the reference's file layout)."""
from __future__ import annotations

import json
import math
import os
import time
from typing import Optional, List, Sequence

import torch

from .. import ops


def split_batch_by_props(batch_size: int, text_prop: float, caption_prop: float, vqa_prop: float):
    """trainer.py:134-154 -> (text, caption, vqa, control) batch sizes.  One torch.multinomial draw over the
    fractional residuals hands out the remainder."""
    control_prop = 1 - text_prop - caption_prop - vqa_prop
    text_bs = int(text_prop * batch_size)
    caption_bs = int(caption_prop * batch_size)
    vqa_bs = int(vqa_prop * batch_size)
    control_bs = int(control_prop * batch_size)
    remainder = batch_size - text_bs - caption_bs - vqa_bs - control_bs
    if remainder > 0:
        residuals = [text_prop * batch_size - text_bs, caption_prop * batch_size - caption_bs,
                     vqa_prop * batch_size - vqa_bs, control_prop * batch_size - control_bs]
        idx = torch.multinomial(torch.tensor(residuals), num_samples=1).item()
        add = [0, 0, 0, 0]
        add[idx] = remainder
        text_bs, caption_bs, vqa_bs, control_bs = text_bs + add[0], caption_bs + add[1], vqa_bs + add[2], control_bs + add[3]
    assert batch_size == text_bs + caption_bs + vqa_bs + control_bs
    return text_bs, caption_bs, vqa_bs, control_bs


def lr_at_step(step: int, *, warmup_steps: int, training_steps: int, base_lr: float, init_lr: float, min_lr: float,
               cosine_decay: bool = True) -> float:
    """schedulers.py:21-32 (the LambdaLR factor times base_lr)."""
    if step <= warmup_steps:
        return init_lr + (base_lr - init_lr) * step / max(1, warmup_steps)
    if cosine_decay:
        progress = (step - warmup_steps) / float(max(1, training_steps - warmup_steps))
        return min_lr + 0.5 * (base_lr - min_lr) * (1 + math.cos(math.pi * progress))
    return base_lr


class FusedAdamW:
    """AdamW + global-norm clip over the policy's flat arenas: one sum-of-squares launch plus one update launch per
    contiguous run of LIVE parameters.  Like torch.optim.AdamW under ``zero_grad(set_to_none=True)`` (what the reference
    runs, train.py:127-133 / trainer.py:186), a parameter whose ``.grad`` is None this cycle is skipped entirely -- no weight
    decay, no moment decay, no step-count increment: ``transformer.wte`` always, the image stack on image-free batches, the
    position tables when disabled, anything frozen.  Step counts (bias correction) are therefore per parameter."""

    def __init__(self, policy, lr, betas=(0.9, 0.95), eps=1e-8, weight_decay=0.1):
        self.policy = policy
        self.lr, self.betas, self.eps, self.weight_decay = lr, betas, eps, weight_decay
        self.exp_avg = torch.zeros_like(policy._param_arena)
        self.exp_avg_sq = torch.zeros_like(policy._param_arena)
        self.sumsq = torch.zeros((), device=policy._param_arena.device)
        self.t = 0              # optimiser steps taken
        self.steps = {}         # per-parameter update count (torch's state['step'])

    def _live_runs(self):
        """[lo, hi, step] arena ranges of the parameters that have a gradient, merged where adjacent with equal counts."""
        p = self.policy
        total = p._param_arena.numel()
        order = p._order
        runs = []
        for k, n in enumerate(order):
            if p._params[n].grad is None:
                continue
            lo = p._offs[n]
            hi = p._offs[order[k + 1]] if k + 1 < len(order) else total
            t = self.steps[n] = self.steps.get(n, 0) + 1
            if runs and runs[-1][1] == lo and runs[-1][2] == t:
                runs[-1][1] = hi
            else:
                runs.append([lo, hi, t])
        return runs

    def step(self, max_norm: float = 0.0, grad_div: float = 1.0):
        p = self.policy
        self.t += 1
        ss = None
        if max_norm > 0:
            # ranges without a gradient hold zeros (GatoPolicy._begin_grads clears them each cycle): the norm over the whole
            # arena equals clip_grad_norm_ over the parameters that have one
            self.sumsq.zero_()
            if getattr(p, "deterministic", False):   # fixed-order sum: the clip factor is bitwise reproducible
                n = p._grad_arena.numel()
                ops.sumsq_ordered(p._grad_arena, self.sumsq, p._buf("ordered_ws", (ops.sumsq_ordered_workspace_bytes(n),), torch.uint8))
            else:
                ops.sumsq(p._grad_arena, self.sumsq)
            ss = self.sumsq
        # the update also rewrites the 16-bit operand copies of the GEMM weights (fp16 forward / bf16 backward), so the
        # next forward starts without a cast kernel
        dual = p.fwd_dtype == torch.float16 and p._w16_arena.dtype == torch.float16
        w16 = p._w16_arena if dual else None
        wbf = p._wbf_arena if dual else (p._w16_arena if p._w16_arena.dtype == torch.bfloat16 and p.fwd_dtype == torch.bfloat16 else None)
        fused = (w16 is not None) or (wbf is not None)
        cast_end = p._cast_end if fused else 0
        for lo, hi, t in self._live_runs():
            nc = max(0, min(hi, cast_end) - lo)
            ops.adamw_step(p._param_arena[lo:hi], p._grad_arena[lo:hi], self.exp_avg[lo:hi], self.exp_avg_sq[lo:hi], self.lr,
                           self.betas[0], self.betas[1], self.eps, self.weight_decay, t, ss, max_norm, grad_div,
                           w_f16=w16[lo:] if (w16 is not None and nc) else None, w_bf16=wbf[lo:] if (wbf is not None and nc) else None,
                           n_cast=nc)
        # the arena was updated in place by raw pointers (no torch version bump): either the copies are fresh (fused) and
        # the recorded versions stay valid, or they must be re-cast by the next forward
        p._bf16_versions = tuple(q._version for q in p._params.values()) if fused else None

    def zero_grad(self):
        self.policy.zero_grad()

    # optimiser state for checkpoint / resume (the reference saves the model only, utils/utils.py:19-32; SURVEY 8(f)4)
    def state_dict(self):
        p = self.policy
        return {"t": self.t, "steps": dict(self.steps), "lr": self.lr, "betas": tuple(self.betas), "eps": self.eps, "weight_decay": self.weight_decay,
                "exp_avg": self.exp_avg.detach().cpu(), "exp_avg_sq": self.exp_avg_sq.detach().cpu(),
                "layout": {n: (int(p._offs[n]), tuple(q.shape)) for n, q in p._params.items()}}

    def load_state_dict(self, sd):
        p = self.policy
        layout = {n: (int(p._offs[n]), tuple(q.shape)) for n, q in p._params.items()}
        if sd["layout"] != layout:
            raise ValueError("optimizer state was saved for a different parameter layout (model configuration)")
        self.t, self.lr = int(sd["t"]), float(sd["lr"])
        self.steps = {n: int(v) for n, v in sd["steps"].items()} if "steps" in sd else {n: self.t for n in layout}
        self.betas, self.eps, self.weight_decay = tuple(sd["betas"]), float(sd["eps"]), float(sd["weight_decay"])
        self.exp_avg.copy_(sd["exp_avg"])
        self.exp_avg_sq.copy_(sd["exp_avg_sq"])


class Trainer:
    def __init__(self, model, optimizer: FusedAdamW, tasks: Sequence, args, sync=None, exp_name: str = "neko_b200"):
        self.model, self.optimizer, self.tasks, self.args, self.sync = model, optimizer, list(tasks), args, sync
        self.exp_name = exp_name
        self.steps = 0
        self.min_lr = args.learning_rate / args.min_factor
        self.prefetch = True          # stage the next batch before reading the current loss (GatoPolicy.stage)
        self._prefetched = None

    # task sampling ----------------------------------------------------------------------------------------
    def _sample(self, kind: str, n: int) -> List[dict]:
        out: List[dict] = []
        tasks = [t for t in self.tasks if t.kind == kind]
        if kind == "control":
            # trainer.py:211-247 draws tasks without replacement until the batch is full
            i = 0
            while len(out) < n and tasks:
                out.extend(tasks[i % len(tasks)].sample_batch(1, max_tokens=self.args.sequence_length))
                i += 1
            return out[:n]
        for t in tasks:
            out.extend(t.sample_batch(n, max_tokens=self.args.sequence_length))
        return out

    def sample_combined_batch(self) -> List[dict]:
        a = self.args
        text_bs, caption_bs, vqa_bs, control_bs = split_batch_by_props(a.batch_size, a.text_prop, a.caption_prop, a.vqa_prop)
        batch: List[dict] = []
        if text_bs > 0:
            batch += self._sample("text", text_bs)
        if caption_bs > 0:
            batch += self._sample("caption", caption_bs)
        if vqa_bs > 0:
            batch += self._sample("vqa", vqa_bs)
        if control_bs > 0:
            batch += self._sample("control", control_bs)
        return batch

    # one optimisation step (trainer.py:127-188) ------------------------------------------------------
    def train_step(self):
        a = self.args
        accum = max(1, a.gradient_accumulation_steps)
        self.optimizer.lr = lr_at_step(self.steps, warmup_steps=a.warmup_steps, training_steps=a.training_steps,
                                       base_lr=a.learning_rate, init_lr=a.init_lr, min_lr=self.min_lr,
                                       cosine_decay=not a.disable_cosine_decay)
        t0 = time.time()
        losses = []
        for micro in range(accum):
            batch = self._prefetched if self._prefetched is not None else self.sample_combined_batch()
            self._prefetched = None
            last = micro == accum - 1
            ctx = self.sync.no_sync() if (self.sync is not None and not last) else _null()
            with ctx:
                _, loss = self.model.forward(inputs=batch, compute_loss=True)
                (loss / accum).backward()
            losses.append(loss.detach().clone())   # graph replays return the same pooled tensor every time
        self.optimizer.step(max_norm=0.0 if a.disable_grad_clip else a.grad_norm_clip)
        self.optimizer.zero_grad()
        self.steps += 1
        if self.prefetch and hasattr(self.model, "stage"):
            # batch producer: sample + plan + enqueue the H2D copy of the next batch while the GPU still works on this step
            self._prefetched = self.model.stage(self.sample_combined_batch(), compute_loss=True)
        loss_val = torch.stack(losses).mean().cpu().item()   # host sync once per step, like trainer.py:188
        return loss_val, {"training/learning_rate": self.optimizer.lr, "time/train_step": time.time() - t0}

    def train(self, steps: int):
        self.model.train()
        logs = []
        for _ in range(steps):
            logs.append(self.train_step())
        return logs


class _null:
    def __enter__(self):
        return self

    def __exit__(self, *a):
        return False


def save_checkpoint(model, save_dir: str, name: str, args, optimizer: Optional["FusedAdamW"] = None, step: Optional[int] = None) -> str:
    """utils/utils.py:19-32 file layout: <save_dir>/<name>.pt (state_dict, loadable by the reference) + args.json; with an
    optimiser also <name>.optim.pt (AdamW moments, step counters) so that training can resume exactly."""
    os.makedirs(save_dir, exist_ok=True)
    path = os.path.join(save_dir, f"{name}.pt")
    torch.save({k: v.detach().cpu() for k, v in model.state_dict().items()}, path)
    with open(os.path.join(save_dir, "args.json"), "w") as f:
        json.dump({k: v for k, v in vars(args).items()}, f, indent=1, default=str)
    if optimizer is not None:
        torch.save({"optimizer": optimizer.state_dict(), "step": step}, os.path.join(save_dir, f"{name}.optim.pt"))
    return path


def load_checkpoint(model, path: str, optimizer: Optional["FusedAdamW"] = None) -> Optional[int]:
    """Inverse of save_checkpoint: strict load of the model, and of the optimiser state when <name>.optim.pt exists.
    Returns the saved step (or None)."""
    sd = torch.load(path, map_location=model.device)
    model.load_state_dict(sd)
    opt_path = path[:-3] + ".optim.pt" if path.endswith(".pt") else path + ".optim.pt"
    step = None
    if optimizer is not None and os.path.exists(opt_path):
        blob = torch.load(opt_path, map_location="cpu", weights_only=False)
        optimizer.load_state_dict(blob["optimizer"])
        step = blob.get("step")
    return step
