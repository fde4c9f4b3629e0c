"""Training loops for the hot path.

train_model           the reference's LID-VAE / LR-VAE loop, lipschitz.py:23-44, same signature.
DataParallelTrainer   one process per GPU: batch sharded by rank, parameters and gradients live in ONE
                      flat fp32 buffer each, a single NCCL all-reduce per step over NVLink, fused Adam
                      (b200vae_adam_step) over the flat buffers.  The path has exactly one exchange
                      step (the gradient all-reduce; SURVEY.md section 8(e)), so nothing else communicates
                      except SyncBatchNorm statistics in the stock encoder.
"""
from __future__ import annotations

import torch
import torch.distributed as dist
from torch import nn

from . import ops
from .utils import apply_grad_clip


def train_model(model, loader, epochs, lr, device, grad_clip=None, wu_strat="linear", wu_start_epoch=0,
                wu_up_amount=None, wu_repeat_interval=10, experiment_logger=None):
    """lipschitz.py:23-44: Adam(lr); per batch forward -> loss -> backward -> clip -> step."""
    model.to(device).train()
    optimizer = torch.optim.Adam(model.parameters(), lr=lr)
    for epoch in range(epochs):
        model.warmup(epoch=epoch, max_epoch=epochs, wu_strat=wu_strat, up_amount=wu_up_amount,
                     start_epoch=wu_start_epoch, repeat_interval=wu_repeat_interval)
        if experiment_logger and hasattr(model, "wu_alpha"):
            experiment_logger.log_alpha_value(epoch, model.wu_alpha)
        for X, _ in loader:
            X = X.to(device)
            optimizer.zero_grad()
            recon, mu, log_var, z_in, z_rec = model(X)
            total_loss, _, _, _ = model.loss(X, recon, mu, log_var, z_in, z_rec)
            total_loss.backward()
            apply_grad_clip(model, grad_clip)
            optimizer.step()
    return model


class _SyncBN1dFn(torch.autograd.Function):
    """Cross-rank BatchNorm1d on [B,C]: ONE all_gather of (mean, biased var, count) in forward and ONE
    all_reduce of (sum dy, sum dy*xhat) in backward -- and, unlike nn.SyncBatchNorm outside graph capture,
    no host synchronisation (its count mask indexing stalls the launch queue once per layer per step)."""

    @staticmethod
    def forward(ctx, x, weight, bias, running_mean, running_var, eps, momentum, training, group):
        world = dist.get_world_size(group)
        n = x.shape[0]
        if training:
            mean_l = x.mean(0)
            var_l = x.var(0, unbiased=False)
            pack = torch.cat([mean_l, var_l, torch.full((1,), float(n), device=x.device, dtype=x.dtype)])
            outs = [torch.empty_like(pack) for _ in range(world)]
            dist.all_gather(outs, pack, group=group)                 # (works on gloo/CPU as well as NCCL)
            allp = torch.stack(outs)
            C = x.shape[1]
            means, vars_, cnt = allp[:, :C], allp[:, C:2 * C], allp[:, 2 * C:]
            N = cnt.sum()
            mean = (means * cnt).sum(0) / N
            var = ((vars_ + (means - mean) ** 2) * cnt).sum(0) / N
            if running_mean is not None:
                with torch.no_grad():
                    running_mean.mul_(1 - momentum).add_(mean, alpha=momentum)
                    running_var.mul_(1 - momentum).add_(var * (N / (N - 1)), alpha=momentum)
        else:
            mean, var, N = running_mean, running_var, torch.tensor(float(n), device=x.device)
        invstd = torch.rsqrt(var + eps)
        xhat = (x - mean) * invstd
        ctx.save_for_backward(xhat, weight, invstd, N.reshape(()))
        ctx.group, ctx.training = group, training
        return xhat * weight + bias

    @staticmethod
    def backward(ctx, dy):
        xhat, weight, invstd, N = ctx.saved_tensors
        dw = (dy * xhat).sum(0)
        db = dy.sum(0)
        if ctx.training:
            sums = torch.stack([db, dw])
            dist.all_reduce(sums, op=dist.ReduceOp.SUM, group=ctx.group)
            dx = (dy - sums[0] / N - xhat * (sums[1] / N)) * (invstd * weight)
        else:
            dx = dy * (invstd * weight)
        return dx, dw, db, None, None, None, None, None, None


class SyncBatchNorm1d(nn.BatchNorm1d):
    """Drop-in for nn.BatchNorm1d on [B,C] inputs (same parameter / buffer names) with cross-rank statistics."""

    def __init__(self, bn: nn.BatchNorm1d, group=None):
        super().__init__(bn.num_features, bn.eps, bn.momentum, bn.affine, bn.track_running_stats)
        self.load_state_dict(bn.state_dict())
        self.to(bn.weight.device)
        self.group = group

    def forward(self, x):
        if x.dim() != 2:
            raise ValueError("SyncBatchNorm1d expects [B, C] inputs")
        if self.training and self.track_running_stats:
            self.num_batches_tracked.add_(1)
        return _SyncBN1dFn.apply(x, self.weight, self.bias, self.running_mean, self.running_var, self.eps,
                                 self.momentum if self.momentum is not None else 0.1, self.training, self.group)


def convert_sync_batchnorm(model, group=None):
    """BatchNorm1d -> SyncBatchNorm1d (lean, works on CPU/gloo too, carries the peer-exchange slots); BatchNorm2d / 3d ->
    nn.SyncBatchNorm, converted child by child so that the SyncBatchNorm1d instances (which ARE _BatchNorm subclasses and
    would be converted back by a whole-model nn.SyncBatchNorm.convert_sync_batchnorm) are left alone."""
    if isinstance(model, (nn.BatchNorm2d, nn.BatchNorm3d)):
        return nn.SyncBatchNorm.convert_sync_batchnorm(model, group)
    for name, child in list(model.named_children()):
        if isinstance(child, SyncBatchNorm1d):
            continue
        if type(child) is nn.BatchNorm1d:
            setattr(model, name, SyncBatchNorm1d(child, group))
        elif isinstance(child, (nn.BatchNorm2d, nn.BatchNorm3d)):
            setattr(model, name, nn.SyncBatchNorm.convert_sync_batchnorm(child, group))
        else:
            convert_sync_batchnorm(child, group)
    return model


class FlatParams:
    """Re-homes every parameter (and its .grad) of `model` as a view into one flat fp32 buffer."""

    def __init__(self, model: nn.Module, alloc=None):
        """`alloc(numel) -> fp32 tensor` supplies the two flat buffers (peer-mapped memory for the fused all-reduce +
        Adam kernel); it may return more elements than asked for (padding stays zero)."""
        params = [p for p in model.parameters() if p.requires_grad]
        if not params:
            raise ValueError("model has no trainable parameters")
        pad4 = lambda k: (k + 3) // 4 * 4        # every parameter starts on a 16-byte boundary (vector loads, TMA, cp.async)
        dev, n = params[0].device, sum(pad4(p.numel()) for p in params)
        self.params = params
        if alloc is None:
            self.flat = torch.zeros(n, dtype=torch.float32, device=dev)        # padding between parameters stays 0
            self.grad = torch.zeros(n, dtype=torch.float32, device=dev)
        else:
            self.flat, self.grad = alloc(n), alloc(n)
            self.flat.zero_(); self.grad.zero_()
        off = 0
        self.views = []
        for p in params:
            k = p.numel()
            self.flat[off:off + k].copy_(p.data.reshape(-1))
            p.data = self.flat[off:off + k].view_as(p.data)
            p.grad = self.grad[off:off + k].view_as(p.data)
            self.views.append(p.grad)
            off += pad4(k)
        self.numel = n
        self._had = [False] * len(params)

    def begin_step(self):
        """Detach every .grad: autograd then hands over each gradient tensor as produced (no zero fill of the flat
        buffer and no accumulate-add launch per parameter); `gather()` moves them into the flat buffer in one launch."""
        for p in self.params:
            p.grad = None

    def gather(self):
        """Copy the step's gradients into the flat buffer with ONE multi-tensor launch and re-attach the views.
        Parameters that received no gradient keep a zero segment."""
        dst, src = [], []
        for i, (p, view) in enumerate(zip(self.params, self.views)):
            g = p.grad
            if g is None:
                if self._had[i]:
                    view.zero_()
                    self._had[i] = False
            elif g.data_ptr() != view.data_ptr():
                dst.append(view); src.append(g)
                self._had[i] = True
            p.grad = view
        if dst:
            torch._foreach_copy_(dst, src)

    def zero_grad(self):
        self.grad.zero_()
        for p, view in zip(self.params, self.views):   # autograd may have replaced .grad; re-attach the views
            if p.grad is None or p.grad.data_ptr() != view.data_ptr():
                p.grad = view


def shard_rows(n_rows, rank, world):
    """Contiguous equal shards (rank r gets rows [r*n/W, (r+1)*n/W)); n must divide evenly so that the
    mean-over-batch losses average exactly across ranks."""
    if n_rows % world:
        raise ValueError(f"global batch {n_rows} is not divisible by world size {world}")
    per = n_rows // world
    return rank * per, (rank + 1) * per


class DataParallelTrainer:
    """Batch-sharded trainer.  `step(x_local, eps_local=None)` runs forward/loss/backward on this rank's
    shard, all-reduces the flat gradient (SUM) once, and applies Adam with grad_scale = 1/world.
    `optimizer_step` can be replaced (tests on CPU/gloo inject a torch implementation; on CUDA the fused
    kernel is used and there is no fallback)."""

    def __init__(self, model, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0, process_group=None,
                 grad_clip=None, sync_bn=True, optimizer_step=None, comm="auto", staged_backward=False,
                 forward_kwargs=None, lr_schedule=None, check_every=256):
        """comm: "peer" = exchanges as kernels over NVLink peer memory (csrc/peer.cuh): BatchNorm statistics inside
        the fused encoder's finalize kernels, gradient all-reduce fused with Adam; "nccl" = torch.distributed
        collectives; "auto" = peer when CUDA IPC mapping works between all ranks, else nccl."""
        # check_every: with the peer-memory exchange, poll the sticky time-out flag every so many steps (one tiny D2H copy
        # + sync) and raise -- a rank that lagged the others by more than the exchange timeout (20 s; eval or checkpointing
        # on one rank only, a stalled data loader) also turns losses / parameters into NaN on the device (csrc/peer.cuh)
        self.check_every = int(check_every) if check_every else 0
        self.world = dist.get_world_size(process_group) if dist.is_initialized() else 1
        self.rank = dist.get_rank(process_group) if dist.is_initialized() else 0
        self.pg = process_group
        # staged_backward: the three-pass backward of main.py:262-284 (latent-recon term first, encoder gradients scaled by
        # 1e-4, then KL, then reconstruction) instead of one total.backward() -- no host sync in it, so the whole staged
        # step still captures into one CUDA graph (the reference's LR-VAE loop is otherwise host bound at its batch sizes)
        self.staged = bool(staged_backward)
        self.forward_kwargs = dict(forward_kwargs or {})       # e.g. {"L": 4}: num_mc_samples of main.py:259
        self.defer_param_grads = True  # False: one-call ICNN backward (the bit-identical reference arm of the tests)
        self._staged = None            # (host tensor, staging slot, copy-done event) of a prefetched batch (step_graphed)
        self._stage = None
        # lr_schedule = ("cosine", T_max): CosineAnnealingLR stepped after every optimiser step (main.py:201-203, 287),
        # evaluated on the device from the step counter so that graph replay follows it (single-GPU / NCCL path)
        if lr_schedule is not None and (lr_schedule[0] != "cosine" or int(lr_schedule[1]) <= 0):
            raise ValueError("lr_schedule must be None or ('cosine', T_max > 0)")
        self.lr_schedule = None if lr_schedule is None else ("cosine", int(lr_schedule[1]))
        if self.world > 1 and sync_bn:
            model = convert_sync_batchnorm(model, process_group)
        self.model = model
        self.peer = None
        on_cuda = next(model.parameters()).is_cuda
        if comm not in ("auto", "peer", "nccl"):
            raise ValueError(f"comm must be auto|peer|nccl, got {comm!r}")
        if self.world > 1 and on_cuda and comm != "nccl" and optimizer_step is None and lr_schedule is None:
            from . import peer as _peer
            self.peer = _peer.PeerComm(process_group) if comm == "peer" else _peer.try_create(process_group)
        self._peer_bufs = None
        if self.peer is not None:
            for mod in model.modules():          # same traversal order on every rank -> same slots
                if isinstance(mod, SyncBatchNorm1d):
                    mod.peer, mod.peer_slots = self.peer, (self.peer.new_slot(), self.peer.new_slot())
            self._adam_slot = self.peer.new_slot(2)
            bufs = []

            def alloc(n):
                b = self.peer.alloc_flat(n)
                bufs.append(b)
                return b.tensor()
            self.fp = FlatParams(model, alloc)
            self._peer_bufs = (bufs[0], bufs[1])          # (parameters, gradients)
        else:
            self.fp = FlatParams(model)
        self.m = torch.zeros_like(self.fp.flat)
        self.v = torch.zeros_like(self.fp.flat)
        self.t = 0
        self.t_dev = torch.zeros((), dtype=torch.int64, device=self.fp.flat.device)   # device step counter (graphs)
        self._graph = None
        self.hp = dict(lr=lr, betas=betas, eps=eps, weight_decay=weight_decay)
        self.grad_clip = grad_clip
        self._opt = optimizer_step or self._fused_adam
        if self.world > 1:   # identical replicas to start from
            dist.broadcast(self.fp.flat, src=0, group=self.pg)
        if self.peer is not None:
            # first peer kernel here, not in the first step: module loading skews the ranks by up to seconds at start-up
            self.peer.barrier()
            torch.cuda.synchronize()
            dist.barrier(group=self.pg)

    def _fused_adam(self, flat, grad, m, v, t, scale, hp):
        # step count kept on the device so that the call is identical every step (CUDA-graph capturable)
        if self.lr_schedule is None:
            ops.adam_step_dev_(flat, grad, m, v, self.t_dev, hp["lr"], hp["betas"], hp["eps"], hp["weight_decay"], scale)
        else:
            ops.adam_step_sched_(flat, grad, m, v, self.t_dev, hp["lr"], hp["betas"], hp["eps"], hp["weight_decay"], scale, 1,
                                 self.lr_schedule[1])

    # ---- whole-step CUDA graph (launch-bound regimes: small batches, multi-GPU with many tiny collectives) ----
    def capture(self, x_example, eps_example=None, warmup=3):
        """Capture forward -> loss -> backward -> all-reduce -> Adam into one CUDA graph.  Optimiser / BatchNorm
        state touched by the warm-up steps is restored, so capturing does not advance training."""
        dev = x_example.device
        self._sx = x_example.clone()
        self._se = None if eps_example is None else eps_example.clone()
        snap = [t.clone() for t in (self.fp.flat, self.m, self.v, self.t_dev)]
        bufs = [(b, b.clone()) for b in self.model.buffers()]
        t_host = self.t
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            for _ in range(warmup):
                self.step(self._sx, self._se)
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize(dev)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            self._sout = self.step(self._sx, self._se)
        for dst, src in zip((self.fp.flat, self.m, self.v, self.t_dev), snap):
            dst.copy_(src)
        for b, old in bufs:
            b.copy_(old)
        self.t = t_host
        self._graph = g
        return self

    def step_graphed(self, x_local, eps_local=None, next_x=None):
        """Replay the captured step on `x_local` (device or pinned host tensor).  `next_x`: the NEXT step's batch, if it is a
        host tensor -- its host-to-device copy is started on a copy stream right away and overlaps this step (a prefetching
        loader in one argument); the next call recognises the tensor and takes the staged copy."""
        if self._graph is None:
            raise RuntimeError("call capture() first")
        cur = torch.cuda.current_stream(self._sx.device)
        if self._staged is not None and x_local is self._staged[0]:
            _, slot, ev = self._staged
            cur.wait_event(ev)
            self._sx.copy_(self._stage[slot], non_blocking=True)
            self._stage_read[slot].record(cur)
        else:
            self._sx.copy_(x_local, non_blocking=True)
        self._staged = None
        if eps_local is not None:
            self._se.copy_(eps_local, non_blocking=True)
        self._graph.replay()
        ops.bump_weights_epoch()          # the replayed Adam kernel changed the weights without any Python running
        if next_x is not None and not next_x.is_cuda:
            self._prefetch(next_x)
        self.t += 1
        self._poll()
        return self._sout

    def _prefetch(self, x_host):
        dev = self._sx.device
        if self._stage is None:
            self._stage = [torch.empty_like(self._sx) for _ in range(2)]
            self._stage_read = [torch.cuda.Event() for _ in range(2)]
            self._copy_stream = torch.cuda.Stream(device=dev)
            self._stage_slot = 0
            for ev in self._stage_read:
                ev.record(torch.cuda.current_stream(dev))
        slot = self._stage_slot = 1 - self._stage_slot
        self._copy_stream.wait_event(self._stage_read[slot])       # the step that last read this staging slot is done with it
        with torch.cuda.stream(self._copy_stream):
            self._stage[slot].copy_(x_host, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(self._copy_stream)
        self._staged = (x_host, slot, ev)

    def _poll(self):
        if self.peer is not None and self.check_every and self.t % self.check_every == 0:
            self.peer.check()

    def step(self, x_local, eps_local=None):
        model, W = self.model, self.world
        self.fp.begin_step()
        kw = dict(self.forward_kwargs)
        if eps_local is not None:
            kw["eps"] = eps_local
        out = model(x_local, **kw)
        total, rec, reg, lr_term = model.loss(x_local, *out)
        det = lambda t: t.detach() if torch.is_tensor(t) else float(t)
        self.last_parts = (det(total), det(rec), det(reg), det(lr_term))     # tensors are static under graph replay
        lr_attached = torch.is_tensor(lr_term) and lr_term.requires_grad
        if self.staged:
            from .main import staged_backward
            # the latent-recon term sums over the batch (Appendix B.2): its global value is the SUM over ranks
            staged_backward(model, total, rec, reg, lr_term * W if (W > 1 and lr_attached) else lr_term)
        else:
            if W > 1 and lr_attached:
                # ... while every other term is a batch mean -> compensate before the 1/W gradient averaging
                total = total + (W - 1) * lr_term
            if total.is_cuda and self.defer_param_grads:
                # the ICNNs' parameter gradients run on a side stream beside the encoder's backward; joined on exit
                with ops.deferred_param_grads():
                    total.backward()
            else:
                total.backward()
        self.fp.gather()
        clip = bool(self.grad_clip and self.grad_clip.get("enabled", False))
        if self.peer is not None and not clip:
            # two-shot all-reduce over peer memory fused with Adam: rank r reduces + updates chunk r and stores it
            # into every replica (csrc/peer.cu); no NCCL call in the step
            self.t += 1
            ops.peer_allreduce_adam_(self.peer, self._adam_slot, self._peer_bufs[1], self._peer_bufs[0], self.m, self.v,
                                     self.fp.flat.numel(), self.t_dev, self.hp["lr"], self.hp["betas"], self.hp["eps"],
                                     self.hp["weight_decay"], 1.0 / W)
            if not torch.cuda.is_current_stream_capturing():
                self._poll()
            return total.detach(), (rec.detach() if torch.is_tensor(rec) else rec), (reg.detach() if torch.is_tensor(reg) else reg)
        if W > 1:
            dist.all_reduce(self.fp.grad, op=dist.ReduceOp.SUM, group=self.pg)
        scale = 1.0 / W
        if self.grad_clip and self.grad_clip.get("enabled", False):
            self.fp.grad.mul_(scale)
            scale = 1.0
            apply_grad_clip(model, self.grad_clip)
        self.t += 1
        self._opt(self.fp.flat, self.fp.grad, self.m, self.v, self.t, scale, self.hp)
        return total.detach(), (rec.detach() if torch.is_tensor(rec) else rec), (reg.detach() if torch.is_tensor(reg) else reg)

    def check(self):
        """Raise if a peer-memory exchange on this rank ever timed out (synchronises; call outside timed regions)."""
        if self.peer is not None:
            self.peer.check()

    @torch.no_grad()
    def global_losses(self, *local_scalars):
        """Mean over ranks of per-rank batch-mean scalars (one tiny all-reduce)."""
        t = torch.stack([torch.as_tensor(s, dtype=torch.float32, device=self.fp.flat.device).reshape(()) for s in local_scalars])
        if self.world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.SUM, group=self.pg)
            t /= self.world
        return t
