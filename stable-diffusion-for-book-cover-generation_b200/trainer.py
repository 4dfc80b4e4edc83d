"""Data-parallel fine-tuning step of the UNet (BASELINE config 3; the loop body of finetune_sd.py:453-494, 569-570):

    noisy = noise_scheduler.add_noise(latents, noise, timesteps)          finetune_sd.py:473-474
    pred  = unet(noisy, timesteps, encoder_hidden_states).sample          finetune_sd.py:480-481
    loss  = F.mse_loss(pred, noise, "none").mean([1,2,3]).mean()          finetune_sd.py:483-484
    accelerator.backward(loss); optimizer.step(); optimizer.zero_grad()   finetune_sd.py:494, 569-570

One process per GPU.  The backward kernels accumulate every parameter gradient into ONE flat fp32 buffer and
complete it from its end towards its start; `BucketReducer` allreduces finished address ranges (NCCL over NVLink,
SUM) while the rest of the backward is still running, and `FlatAdamW` does the whole optimizer step -- gradient
averaging, AdamW, the bf16 re-cast of the weights and the zeroing of the gradients -- in one pass over the flat
buffers.  Gradient accumulation (`sync=False` micro-steps, accelerate's no_sync, finetune_sd.py:454-458) simply
skips the reduction: the kernels keep accumulating.
"""
from __future__ import annotations

import torch
import torch.distributed as dist

from . import ops


class BucketReducer:
    """Allreduce of a flat gradient buffer in address ranges that become final back to front.

    on_ready(offset) announces that flat[offset:] is final; whenever at least `bucket_bytes` are pending (or offset
    reaches 0) the pending range is reduced asynchronously.  finish() waits for all of them."""

    def __init__(self, flat: torch.Tensor, group=None, bucket_bytes: int = 64 << 20):
        self.flat, self.group, self.bucket_bytes = flat, group, int(bucket_bytes)
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.esize = flat.element_size()
        self.begin()

    def begin(self):
        self.hi = self.flat.numel()
        self.works = []
        self.ranges = []

    def on_ready(self, offset: int):
        if offset >= self.hi:
            return
        if (self.hi - offset) * self.esize >= self.bucket_bytes or offset == 0:
            self._launch(offset, self.hi)
            self.hi = offset

    def _launch(self, a: int, b: int):
        self.ranges.append((a, b))
        if self.world > 1:
            self.works.append(dist.all_reduce(self.flat[a:b], op=dist.ReduceOp.SUM, group=self.group, async_op=True))

    def finish(self, wait=True):
        """Launch the allreduce of whatever is still pending; wait=False leaves the waiting to the caller (Trainer interleaves it
        with the optimizer: `pending()` yields (range, work) in launch order)."""
        if self.hi > 0:
            self._launch(0, self.hi)
            self.hi = 0
        if wait:
            for w in self.works:
                w.wait()
            self.works = []

    def pending(self):
        """(a, b, work) of every launched range, in launch order (= completion order on the NCCL stream); clears the list"""
        out = [(a, b, w) for (a, b), w in zip(self.ranges, self.works)] if self.works else [(a, b, None) for a, b in self.ranges]
        self.works = []
        return out


class FlatAdamW(torch.optim.Optimizer):
    """torch.optim.AdamW semantics over train.FlatParams (one fused kernel per step).

    It IS a `torch.optim.Optimizer` (one param group over the flat fp32 master buffer), so the reference's
    `torch.optim.lr_scheduler.CosineAnnealingLR(optimizer, T_max=..., eta_min=1e-6)` + `scheduler.step()` after every
    `optimizer.step()` (finetune_sd.py:421-422, 577) drives it unchanged: the kernel reads `param_groups[0]["lr"]` at every step;
    `state_dict()` / `load_state_dict()` carry the moments and the step count.  When the model's flat buffers are rebuilt
    (`unet.to()` un-homes the parameters) the trainers `rebind()` this object instead of replacing it, so a scheduler that holds
    a reference to it stays attached."""

    def __init__(self, flat, lr=1e-5, betas=(0.9, 0.999), eps=1e-8, weight_decay=1e-2, state=None):
        if lr < 0 or eps < 0 or weight_decay < 0 or not (0 <= betas[0] < 1 and 0 <= betas[1] < 1):
            raise ValueError(f"invalid AdamW hyper-parameters lr={lr} betas={betas} eps={eps} weight_decay={weight_decay}")
        super().__init__([flat.master], dict(lr=lr, betas=tuple(betas), eps=eps, weight_decay=weight_decay))
        self.flat = None
        self.rebind(flat, state)

    def rebind(self, flat, state=None):
        """(re)attach to a FlatParams: same model and layout -> the moments and the step count carry over (from `state`, another
        FlatAdamW, or from this object's own state) instead of silently restarting from zero"""
        old = state.state.get(state.flat.master) if state is not None else (
            self.state.pop(self.flat.master, None) if self.flat is not None else None)
        self.flat = flat
        self.param_groups[0]["params"] = [flat.master]
        self.state.clear()
        self.state[flat.master] = self._make_state(flat, old)
        # contiguous runs of TRAINABLE regions: frozen parameters (requires_grad=False) get neither an update nor
        # decoupled weight decay, as with torch.optim.AdamW over `filter(requires_grad, parameters)`
        self.spans = []
        for r in flat.order:
            if not r.param.requires_grad:
                continue
            a, b = r.off, r.off + (r.numel + 63) // 64 * 64
            if self.spans and self.spans[-1][1] == a:
                self.spans[-1][1] = b
            else:
                self.spans.append([a, b])
        if self.spans:
            self.spans[-1][1] = min(self.spans[-1][1], flat.master.numel())
        return self

    def _make_state(self, flat, old):
        dev = flat.master.device
        if old is not None and "exp_avg" in old and old["exp_avg"].numel() == flat.master.numel():
            return dict(step=int(old["step"]), exp_avg=old["exp_avg"].to(dev), exp_avg_sq=old["exp_avg_sq"].to(dev))
        return dict(step=0, exp_avg=torch.zeros_like(flat.master), exp_avg_sq=torch.zeros_like(flat.master))

    # the hyper-parameters live in param_groups[0] (what torch's lr schedulers write); attribute access for the callers
    lr = property(lambda self: self.param_groups[0]["lr"], lambda self, v: self.param_groups[0].__setitem__("lr", v))
    betas = property(lambda self: self.param_groups[0]["betas"], lambda self, v: self.param_groups[0].__setitem__("betas", tuple(v)))
    eps = property(lambda self: self.param_groups[0]["eps"], lambda self, v: self.param_groups[0].__setitem__("eps", v))
    weight_decay = property(lambda self: self.param_groups[0]["weight_decay"],
                            lambda self, v: self.param_groups[0].__setitem__("weight_decay", v))
    exp_avg = property(lambda self: self.state[self.flat.master]["exp_avg"])
    exp_avg_sq = property(lambda self: self.state[self.flat.master]["exp_avg_sq"])
    steps = property(lambda self: self.state[self.flat.master]["step"],
                     lambda self, v: self.state[self.flat.master].__setitem__("step", int(v)))

    _state_dtypes = {"exp_avg": torch.float32, "exp_avg_sq": torch.float32}

    def load_state_dict(self, state_dict):
        # validated BEFORE anything is replaced: a state that does not fit leaves this optimizer as it was
        want = {k: v.shape for k, v in self.state[self.flat.master].items() if torch.is_tensor(v)}
        saved = state_dict["state"].get(0, {})
        for k, shape in want.items():
            v = saved.get(k)
            if not torch.is_tensor(v) or v.shape != shape:
                raise ValueError(f"optimizer state '{k}' does not fit this model's flat parameter buffer ({tuple(shape)})")
            if v.dtype != self._state_dtypes[k]:
                raise ValueError(f"optimizer state '{k}' was saved as {v.dtype}, expected {self._state_dtypes[k]}")
        super().load_state_dict(state_dict)       # torch casts every state tensor to the parameter's dtype (u8 codes included)
        st = self.state[self.flat.master]
        st["step"] = int(st["step"])
        for k in want:
            st[k] = st[k].to(device=self.flat.master.device, dtype=self._state_dtypes[k]).contiguous()

    def zero_grad(self, set_to_none: bool = True):
        """`optimizer.zero_grad()` of the reference loop (finetune_sd.py:570).  step() already zeroes the flat gradient buffer in the
        same pass that consumes it; this is for callers that discard gradients without stepping."""
        if self.flat.grad is not None:
            self.flat.zero_grad()

    def _update(self, a, b, grad_scale, zero_grad):
        f = self.flat
        ops.adamw_step(f.master[a:b], f.grad[a:b], self.exp_avg[a:b], self.exp_avg_sq[a:b], f.wb[a:b], self.lr, self.betas[0],
                       self.betas[1], self.eps, self.weight_decay, self.steps, grad_scale=grad_scale, zero_grad=zero_grad)

    def begin_step(self):
        """open an optimizer step that is applied range by range (step_range), e.g. as gradient buckets finish their allreduce"""
        self.steps += 1

    def step_range(self, lo, hi, grad_scale=1.0, zero_grad=True):
        """the part of the current step (begin_step) that falls into flat[lo:hi): trainable spans clipped to the range"""
        for a, b in self.spans:
            a2, b2 = max(a, lo), min(b, hi)
            if a2 < b2:
                self._update(a2, b2, grad_scale, zero_grad)

    def end_step(self):
        self.flat.model.mark_weights_changed()
        self._opt_called = True      # what torch's lr schedulers look at to tell "optimizer stepped before scheduler.step()"
        return self

    def step(self, closure=None, grad_scale=1.0, zero_grad=True):
        if closure is not None:
            raise NotImplementedError("FlatAdamW.step takes no closure (the reference never passes one)")
        self.steps += 1
        for a, b in self.spans:
            self._update(a, b, grad_scale, zero_grad)
        # the kernel wrote the bf16 copy itself: the version bookkeeping of refresh_weights() stays valid.  The raw kernel
        # bumps no tensor version, so tell the facade: its inference engines hold their own packed copy of the weights and
        # must repack before the next eval-mode forward (finetune_sd.py:264-271 samples between training steps).
        self.flat.model.mark_weights_changed()
        return self


def create_dynamic_map(signed: bool = True, n: int = 7) -> torch.Tensor:
    """bitsandbytes' "dynamic" 8-bit code book (functional.create_dynamic_map, 0.35.x): 256 sorted fp32 values; decade i of the
    7 decades 1e-6 .. 1 holds 2^i (signed: of each sign) / 2^(i+1) (unsigned) linearly spaced fractions, plus 0 and 1."""
    data = []
    extra = (2 ** (7 - n) - 1) * (1 if signed else 2)
    for i in range(n):
        items = 2 ** (i + 7 - n) + 1 if signed else 2 ** (i + 7 - n + 1) + 1
        edges = torch.linspace(0.1, 1, items)
        means = (edges[:-1] + edges[1:]) / 2.0
        data += ((10 ** (-(n - 1) + i)) * means).tolist()
        if signed:
            data += (-(10 ** (-(n - 1) + i)) * means).tolist()
    if extra > 0:
        edges = torch.linspace(0.1, 1, extra + 1)
        means = (edges[:-1] + edges[1:]) / 2.0
        data += ((10 ** (-(n - 1) + i)) * means).tolist()
        if signed:
            data += (-(10 ** (-(n - 1) + i)) * means).tolist()
    data += [0.0, 1.0]
    if len(data) != 256:
        raise ValueError("the 8-bit code book must have 256 entries")
    return torch.tensor(sorted(data), dtype=torch.float32)


class FlatAdamW8bit(FlatAdamW):
    """`bnb.optim.AdamW8bit(params, lr, weight_decay, min_8bit_size=16384)` -- the reference's DEFAULT optimizer
    (finetune_sd.py:300 use_8bit_adam=True, :407-420) -- over train.FlatParams, one fused kernel per step
    (csrc/optim8bit.cu: b200sd_adamw8bit_step).

    Both Adam moments are 1-byte codes of bitsandbytes' dynamic code books with one fp32 absmax per block of 2048 values;
    tensors with fewer than `min_8bit_size` elements (biases, norms) keep fp32 moments in a compact side buffer, frozen
    parameters are skipped.  2 B of optimizer state per parameter instead of 8 B, and 18 B (22 B with the gradient zeroing)
    of HBM traffic per parameter and step instead of 30 B (34 B).  Blocks run over the flat buffer, not per tensor (a block may
    hold the tail of one tensor and the head of the next); the update order is bitsandbytes' (decay after the Adam update).
    It is a torch.optim.Optimizer like FlatAdamW: lr schedulers, state_dict(), rebind() work the same way."""

    BLOCK, CHUNK, MODE_8BIT, MODE_SKIP = 2048, 64, -1, -2
    _state_dtypes = {"state1": torch.uint8, "state2": torch.uint8, "absmax1": torch.float32, "absmax2": torch.float32,
                     "exp_avg": torch.float32, "exp_avg_sq": torch.float32}

    def __init__(self, flat, lr=1e-5, betas=(0.9, 0.999), eps=1e-8, weight_decay=1e-2, min_8bit_size=16384, state=None):
        self.min_8bit_size = int(min_8bit_size)
        self._pending = False
        super().__init__(flat, lr=lr, betas=betas, eps=eps, weight_decay=weight_decay, state=state)

    def _make_state(self, flat, old):
        dev, n = flat.master.device, flat.master.numel()
        if n % self.CHUNK:
            raise ValueError("the flat parameter buffer must be a multiple of 64 elements")
        mode = torch.full((n // self.CHUNK,), self.MODE_SKIP, dtype=torch.int32)
        n_small = 0
        for r in flat.order:
            c0, c1 = r.off // self.CHUNK, (r.off + r.numel + self.CHUNK - 1) // self.CHUNK
            if not r.param.requires_grad:
                continue
            if r.numel < self.min_8bit_size:
                mode[c0:c1] = torch.arange(n_small, n_small + (c1 - c0) * self.CHUNK, self.CHUNK, dtype=torch.int32)
                n_small += (c1 - c0) * self.CHUNK
            else:
                mode[c0:c1] = self.MODE_8BIT
        self.chunk_mode = mode.to(dev)
        self.qmap1, self.qmap2 = create_dynamic_map(True).to(dev), create_dynamic_map(False).to(dev)
        nblocks = (n + self.BLOCK - 1) // self.BLOCK
        n_small = max(n_small, self.CHUNK)            # never an empty (null-pointer) buffer
        if (old is not None and "state1" in old and old["state1"].numel() == n and old["exp_avg"].numel() == n_small):
            return {k: (int(v) if k == "step" else v.to(dev)) for k, v in old.items()}
        return dict(step=0, state1=torch.zeros(n, dtype=torch.uint8, device=dev), state2=torch.zeros(n, dtype=torch.uint8, device=dev),
                    absmax1=torch.zeros(nblocks, device=dev), absmax2=torch.zeros(nblocks, device=dev),
                    exp_avg=torch.zeros(n_small, device=dev), exp_avg_sq=torch.zeros(n_small, device=dev))

    def state_bytes(self):
        return sum(v.numel() * v.element_size() for v in self.state[self.flat.master].values() if torch.is_tensor(v))

    def _launch(self, grad_scale, zero_grad):
        f, st = self.flat, self.state[self.flat.master]
        ops.adamw8bit_step(f.master, f.grad, st["state1"], st["state2"], st["absmax1"], st["absmax2"], self.qmap1, self.qmap2,
                           self.chunk_mode, st["exp_avg"], st["exp_avg_sq"], f.wb, self.lr, self.betas[0], self.betas[1], self.eps,
                           self.weight_decay, self.steps, grad_scale=grad_scale, zero_grad=zero_grad)

    # a quantisation block of 2048 values does not respect gradient-bucket boundaries: the range-by-range form of the step
    # (Trainer's pipelined AdamW) is accepted and applied as ONE launch when the step is closed
    def begin_step(self):
        self.steps += 1
        self._pending = None

    def step_range(self, lo, hi, grad_scale=1.0, zero_grad=True):
        if self._pending not in (None, (grad_scale, zero_grad)):
            raise ValueError("FlatAdamW8bit: the ranges of one step must share grad_scale / zero_grad")
        self._pending = (grad_scale, zero_grad)

    def end_step(self):
        if self._pending:
            self._launch(*self._pending)
        self._pending = False
        return super().end_step()

    def step(self, closure=None, grad_scale=1.0, zero_grad=True):
        if closure is not None:
            raise NotImplementedError("FlatAdamW8bit.step takes no closure (the reference never passes one)")
        self.steps += 1
        self._launch(grad_scale, zero_grad)
        self.flat.model.mark_weights_changed()
        return self


def _make_optimizer(flat, optim_bits, opt_args, min_8bit_size):
    if optim_bits == 32:
        return FlatAdamW(flat, **opt_args)
    if optim_bits == 8:
        return FlatAdamW8bit(flat, min_8bit_size=min_8bit_size, **opt_args)
    raise ValueError("optim_bits must be 32 (torch.optim.AdamW semantics) or 8 (bnb.optim.AdamW8bit semantics)")


class Trainer:
    def __init__(self, unet, noise_scheduler, lr=1e-5, betas=(0.9, 0.999), eps=1e-8, weight_decay=1e-2, group=None,
                 bucket_bytes: int = 64 << 20, optim_bits: int = 32, min_8bit_size: int = 16384):
        """optim_bits=8: the reference's default `bnb.optim.AdamW8bit(..., min_8bit_size=16384)` (finetune_sd.py:300, 407-410) as
        FlatAdamW8bit; 32 (default here): torch.optim.AdamW semantics, the reference's use_8bit_adam=False branch."""
        self.optim_bits, self.min_8bit_size = optim_bits, min_8bit_size
        self.unet, self.sched, self.group = unet.train(), noise_scheduler, group
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.bucket_bytes = bucket_bytes
        self.opt_args = dict(lr=lr, betas=betas, eps=eps, weight_decay=weight_decay)
        unet.enable_direct_gradients()
        self.reducer = None
        self.opt = None
        self.micro_steps = 0
        self.allreduce_enabled = True    # False: every rank steps on its local gradient (bench.py times the exposed communication)

    def _prepare(self, device):
        from .autograd import ensure_flat
        flat = ensure_flat(self.unet, device)
        if self.reducer is None or self.reducer.flat is not flat.grad:
            self.reducer = BucketReducer(flat.grad, self.group, self.bucket_bytes)
            self.opt = (_make_optimizer(flat, self.optim_bits, self.opt_args, self.min_8bit_size) if self.opt is None
                        else self.opt.rebind(flat))
            flat.zero_grad()
            flat.attach_grads()
            self.micro_steps = 0

    def optimizer(self, device=None):
        """the FlatAdamW of this trainer (a torch.optim.Optimizer), e.g. to hang the reference's lr scheduler on it:
        `sched = torch.optim.lr_scheduler.CosineAnnealingLR(trainer.optimizer(), T_max=n, eta_min=1e-6)`; call `sched.step()` after
        every `train_step(sync=True)` (finetune_sd.py:421-422, 577)."""
        self._prepare(device if device is not None else self.unet.device)
        return self.opt

    def train_step(self, latents, noise, timesteps, encoder_hidden_states, sync=True):
        """one micro-step; with sync=True (the default) also allreduce + optimizer step.  Returns the loss (0-d tensor).
        Gradient accumulation follows accelerate (finetune_sd.py:454-458, 494): the k micro-steps since the last optimizer
        step are AVERAGED (accelerator.backward divides the loss by gradient_accumulation_steps), and so are the ranks."""
        unet = self.unet
        self._prepare(latents.device)
        reduce_now = sync and self.world > 1 and self.allreduce_enabled
        if reduce_now:
            self.reducer.begin()
        unet._grad_ready_hook = self.reducer.on_ready if reduce_now else None
        noisy = self.sched.add_noise(latents, noise, timesteps)
        pred = unet(noisy, timesteps, encoder_hidden_states).sample
        loss = ops.mse_loss(pred, noise)
        loss.backward()
        unet._grad_ready_hook = None
        self.micro_steps += 1
        if sync:
            scale = 1.0 / (self.world * self.micro_steps)
            if reduce_now:
                # AdamW bucket by bucket, in the order the buckets were put on the wire: the update of the early buckets (the
                # tail of the flat buffer, reduced while the backward was still running) overlaps the allreduce of the last
                # ones, which used to be fully exposed; work.wait() makes the compute STREAM wait, not the host
                self.reducer.finish(wait=False)
                self.opt.begin_step()
                for a, b, work in self.reducer.pending():
                    if work is not None:
                        work.wait()
                    self.opt.step_range(a, b, grad_scale=scale, zero_grad=True)
                self.opt.end_step()
            else:
                self.opt.step(grad_scale=scale, zero_grad=True)
            self.micro_steps = 0
        return loss.detach()


def allreduce_in_chunks(flat: torch.Tensor, chunks: int, group=None):
    """SUM-allreduce a flat buffer as `chunks` asynchronous pieces (the first is on the wire while the host queues the rest);
    returns the (begin, end) ranges it used.  A world of 1 reduces nothing."""
    n = flat.numel()
    step = (n + max(1, int(chunks)) - 1) // max(1, int(chunks))
    ranges = [(a, min(a + step, n)) for a in range(0, n, step)]
    if dist.is_initialized() and dist.get_world_size(group) > 1:
        works = [dist.all_reduce(flat[a:b], op=dist.ReduceOp.SUM, group=group, async_op=True) for a, b in ranges]
        for w in works:
            w.wait()
    return ranges


class TextEncoderTrainer:
    """Data-parallel fine-tuning step of the TEXT ENCODER with the UNet frozen (BASELINE config 4; the reference's default mode,
    finetune_sd.py:29, 375-383, 391-395, 477-494):

        ctx   = text_encoder(input_ids)[0]                                     finetune_sd.py:477   (b200sd.clip.CLIPTextModel)
        noisy = noise_scheduler.add_noise(latents, noise, timesteps)           finetune_sd.py:473-474
        pred  = unet(noisy, timesteps, ctx).sample                             finetune_sd.py:480-481 (frozen: forward + data
        loss  = mse(pred, noise); accelerator.backward(loss); optimizer.step()                         gradient down to ctx)

    The UNet's backward hands d(loss)/d(ctx) to the text encoder's backward plan, whose kernels accumulate all 123 M parameter
    gradients into ONE flat fp32 buffer; that buffer is allreduced over NCCL in `chunks` pieces (the first starts while the host
    is still queueing the others) and `FlatAdamW` updates master weights, the bf16 tensor-core copy and zeroes the gradients in
    one pass."""

    def __init__(self, text_encoder, unet, noise_scheduler, lr=1e-5, betas=(0.9, 0.999), eps=1e-8, weight_decay=1e-2, group=None,
                 chunks: int = 4, optim_bits: int = 32, min_8bit_size: int = 16384):
        self.optim_bits, self.min_8bit_size = optim_bits, min_8bit_size
        self.te, self.unet, self.sched, self.group = text_encoder.train(), unet.eval().requires_grad_(False), noise_scheduler, group
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.opt_args = dict(lr=lr, betas=betas, eps=eps, weight_decay=weight_decay)
        self.chunks = max(1, int(chunks))
        text_encoder.enable_direct_gradients()
        self.opt = None
        self._flat_id = None
        self.micro_steps = 0
        self.allreduce_enabled = True

    def _prepare(self, device):
        flat = self.te._ensure_flat(device)
        if self._flat_id is not flat.grad:
            self.opt = (_make_optimizer(flat, self.optim_bits, self.opt_args, self.min_8bit_size) if self.opt is None
                        else self.opt.rebind(flat))
            flat.zero_grad()
            flat.attach_grads()
            self._flat_id = flat.grad
            self.micro_steps = 0
        return flat

    def optimizer(self, device=None):
        """the FlatAdamW of this trainer (see Trainer.optimizer)"""
        self._prepare(device if device is not None else self.te.device)
        return self.opt

    def train_step(self, latents, noise, timesteps, input_ids, sync=True):
        flat = self._prepare(latents.device)
        ctx = self.te(input_ids)[0]
        noisy = self.sched.add_noise(latents, noise, timesteps)
        pred = self.unet(noisy, timesteps, ctx).sample
        loss = ops.mse_loss(pred, noise)
        loss.backward()
        self.micro_steps += 1
        if sync:
            if self.world > 1 and self.allreduce_enabled:
                allreduce_in_chunks(flat.grad, self.chunks, self.group)
            self.opt.step(grad_scale=1.0 / (self.world * self.micro_steps), zero_grad=True)
            self.micro_steps = 0
        return loss.detach()
