"""Multi-GPU plumbing for the forward path: one process per GPU, batch rows (sequences) sharded across ranks.

Sequences are independent units -- frames only interact through the per-sequence KV memory, which lives on the rank that
owns the sequence (SURVEY.md section 8e) -- so the data path needs NO collective.  `all_gather_rows` is an optional convenience
for a caller that wants every rank's actions / logits in one place."""
import torch
import torch.distributed as dist


def shard_range(batch: int, rank: int, world: int):
    """Contiguous [lo, hi) slice of the batch rows owned by `rank` (sizes differ by at most one)."""
    base, rem = divmod(batch, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def all_gather_rows(x: torch.Tensor, batch: int) -> torch.Tensor:
    """Concatenates the per-rank row shards of `x` (dim 0) on every rank; works for uneven shards."""
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        return x
    world = dist.get_world_size()
    sizes = [shard_range(batch, r, world) for r in range(world)]
    pad = max(hi - lo for lo, hi in sizes)
    buf = torch.zeros((pad,) + tuple(x.shape[1:]), dtype=x.dtype, device=x.device)
    buf[: x.shape[0]] = x
    outs = [torch.empty_like(buf) for _ in range(world)]
    dist.all_gather(outs, buf)
    return torch.cat([o[: hi - lo] for o, (lo, hi) in zip(outs, sizes)], dim=0)


class HostFramePipe:
    """Double-buffered pinned-host -> device upload of (frames, first) chunks on a side stream, so that the upload of chunk
    i+1 overlaps the forward of chunk i (the forward itself never waits on the host).  Usage:

        pipe = HostFramePipe(device)
        pipe.submit(host_img, host_first)            # starts the async copy of the first chunk
        for ...:
            img, first = pipe.take()                 # device tensors of the chunk submitted last; compute stream waits on the copy
            pipe.submit(next_host_img, next_host_first)
            out, state = policy({"img": img}, first, state)
    """

    def __init__(self, device):
        self.device = torch.device(device)
        self.stream = torch.cuda.Stream(device=self.device)
        self.slots = [None, None]
        self.events = [None, None]
        self.cur = 0
        self.pending = None

    def submit(self, host_img: torch.Tensor, host_first: torch.Tensor):
        i = self.cur
        # slot i was last read by the forward of two chunks ago, already enqueued on the compute stream: order the overwrite after it
        self.stream.wait_stream(torch.cuda.current_stream(self.device))
        if self.slots[i] is None or self.slots[i][0].shape != host_img.shape:
            # static device slots (allocated once): no allocator traffic, no implicit synchronisation in the steady state
            self.slots[i] = (torch.empty(host_img.shape, dtype=host_img.dtype, device=self.device),
                             torch.empty(host_first.shape, dtype=host_first.dtype, device=self.device))
        with torch.cuda.stream(self.stream):
            self.slots[i][0].copy_(host_img, non_blocking=True)
            self.slots[i][1].copy_(host_first, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(self.stream)
        self.events[i] = ev
        self.pending = i
        self.cur ^= 1

    def take(self):
        if self.pending is None:
            raise RuntimeError("HostFramePipe.take() before any submit()")
        i = self.pending
        torch.cuda.current_stream(self.device).wait_event(self.events[i])
        return self.slots[i]


class FlatAdamDP:
    """Data-parallel optimizer plumbing of the BC step (SURVEY section 8e, behavioural_cloning.py:63-67,119-123), independent of how the
    gradients are produced: all parameters are re-pointed into ONE flat fp32 bucket, their `.grad`s into a second flat bucket,
    so that a step is  one NCCL all-reduce (sum) over the gradient bucket  +  one fused Adam kernel (`vpt_adam_step`,
    torch.optim.Adam semantics with L2 weight decay; 1/world_size folded into the kernel).

    Pass only the parameters that receive a gradient (behavioural cloning: everything but `value_head.*`, whose `.grad` stays None in
    the reference; the RL step, training.RLTrainer: every parameter with requires_grad, `value_head.linear.*` included -- the return
    normaliser's buffers are requires_grad=False and stay out of the bucket): torch.optim.Adam SKIPS a parameter without a gradient
    (no weight decay, no moment update), whereas a slice of this
    bucket that is never written would still be decayed.  `step()` therefore refuses parameters whose `.grad` no longer aliases the
    bucket (e.g. after `zero_grad(set_to_none=True)` on the module) instead of silently applying Adam to zeros."""

    def __init__(self, params, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0):
        self.params = [p for p in params if p.requires_grad]
        dev = self.params[0].device
        sizes = [(p.numel() + 3) // 4 * 4 for p in self.params]  # 16-byte aligned slices
        self.n = sum(sizes)
        self.flat_p = torch.zeros(self.n, dtype=torch.float32, device=dev)
        self.flat_g = torch.zeros(self.n, dtype=torch.float32, device=dev)
        self.exp_avg = torch.zeros_like(self.flat_p)
        self.exp_avg_sq = torch.zeros_like(self.flat_p)
        off = 0
        with torch.no_grad():
            for p, sz in zip(self.params, sizes):
                view = self.flat_p[off:off + p.numel()].view_as(p)
                view.copy_(p)
                p.data = view                                        # parameters now alias the flat bucket
                p.grad = self.flat_g[off:off + p.numel()].view_as(p)  # and so do their gradients
                off += sz
        self.lr, self.betas, self.eps, self.weight_decay, self.t = lr, betas, eps, weight_decay, 0
        self._pending = None  # (lo, hi, work) of a gradient slice whose all-reduce is already in flight

    def zero_grad(self):
        if self._pending is not None:  # a step that raised after `reduce_async` left a collective in flight: finish it first
            self._pending[2].wait()
            self._pending = None
        self.flat_g.zero_()

    def state_dict(self):
        """Moments, step count and hyper-parameters (CPU tensors); the bucket layout is implied by the parameter order."""
        return {"step": self.t, "n": self.n, "exp_avg": self.exp_avg.detach().cpu().clone(), "exp_avg_sq": self.exp_avg_sq.detach().cpu().clone(),
                "lr": self.lr, "betas": tuple(self.betas), "eps": self.eps, "weight_decay": self.weight_decay}

    def load_state_dict(self, sd):
        if sd["n"] != self.n:
            raise ValueError(f"FlatAdamDP: bucket size {sd['n']} in the checkpoint != {self.n} (different parameter set)")
        self.exp_avg.copy_(sd["exp_avg"])
        self.exp_avg_sq.copy_(sd["exp_avg_sq"])
        self.t = int(sd["step"])
        self.lr, self.betas, self.eps, self.weight_decay = sd["lr"], tuple(sd["betas"]), sd["eps"], sd["weight_decay"]

    def offset_of(self, param) -> int:
        """Start of `param`'s slice in the flat buckets (the bucket follows the order of the parameter list)."""
        return (param.data_ptr() - self.flat_p.data_ptr()) // self.flat_p.element_size()

    def reduce_async(self, lo: int, hi: int) -> None:
        """Start the all-reduce of gradient slice [lo, hi) now -- its gradients are final -- and keep computing: the collective runs
        on the process group's own stream behind the work already enqueued, `step()` waits for it and reduces the rest.  Used to hide
        the bulk of the bucket (transformer, heads, dense: ~98 % of the parameters, finished ~15 % into the backward pass) behind
        the ImpalaCNN backward (SURVEY section 8e: "launched once after backward, or overlapped with the stack-0 wgrad tail")."""
        world = dist.get_world_size() if (dist.is_available() and dist.is_initialized()) else 1
        if world == 1 or hi <= lo:
            return
        if self._pending is not None:
            raise RuntimeError("FlatAdamDP.reduce_async: one slice per step")
        work = dist.all_reduce(self.flat_g[lo:hi], op=dist.ReduceOp.SUM, async_op=True)
        self._pending = (lo, hi, work)

    def reduce_gradients(self) -> int:
        """The gradient all-reduce (sum) of the BC step: ONE collective over the flat bucket, or -- after `reduce_async` -- the
        remaining slices plus a wait on the one already in flight.  Returns the world size (the mean is folded into the Adam kernel)."""
        world = dist.get_world_size() if (dist.is_available() and dist.is_initialized()) else 1
        if world > 1:
            if self._pending is None:
                dist.all_reduce(self.flat_g, op=dist.ReduceOp.SUM)
            else:
                lo, hi, work = self._pending
                self._pending = None
                if lo > 0:
                    dist.all_reduce(self.flat_g[:lo], op=dist.ReduceOp.SUM)
                if hi < self.n:
                    dist.all_reduce(self.flat_g[hi:], op=dist.ReduceOp.SUM)
                work.wait()
        return world

    def clip_grad_norm_(self, max_norm: float, world: int = 1):
        """`th.nn.utils.clip_grad_norm_` over the whole (already reduced) bucket, without a host sync.  NOTE: the reference's own call
        (behavioural_cloning.py:119) is a no-op -- it passes the `policy.parameters()` generator that the Adam constructor has
        already exhausted -- so `step()` does not clip unless asked to."""
        total = torch.linalg.vector_norm(self.flat_g) / world
        coef = torch.clamp(max_norm / (total + 1e-6), max=1.0)
        self.flat_g.mul_(coef)
        return total

    def step(self, max_grad_norm=None):
        base = self.flat_g.data_ptr()
        for p in self.params:
            if p.grad is None or not (base <= p.grad.data_ptr() < base + self.flat_g.numel() * 4):
                raise RuntimeError("FlatAdamDP.step: a parameter's .grad no longer aliases the flat gradient bucket (use FlatAdamDP.zero_grad(), "
                                   "not module.zero_grad(set_to_none=True))")
        world = self.reduce_gradients()
        if max_grad_norm is not None:
            self.clip_grad_norm_(max_grad_norm, world)
        self.t += 1
        if self.flat_p.is_cuda:
            from . import _native as nat
            nat.check(nat.lib().vpt_adam_step(self.flat_p.data_ptr(), self.flat_g.data_ptr(), self.exp_avg.data_ptr(),
                                              self.exp_avg_sq.data_ptr(), self.n, self.lr, self.betas[0], self.betas[1], self.eps,
                                              self.weight_decay, 1.0 / world, self.t, torch.cuda.current_stream().cuda_stream),
                      "vpt_adam_step")
            # the kernel wrote the parameters through raw pointers: bump their version counters so that the kernel-layout weight
            # copies (policy._Prepared, training.BCTrainer._weights) are rebuilt before the next forward
            for p in self.params:
                torch.autograd.graph.increment_version(p)
        else:
            raise RuntimeError("FlatAdamDP.step: the fused Adam kernel is CUDA only (no CPU fallback)")
