"""Training step driver for the CTR zoo: streams, CUDA graph, end-to-end input pipeline.

One step = H2D(ids, dense, labels) -> sparse pull (peer loads) -> dense fwd/bwd ->
fused sparse push+update (P2P dispatch, combine, optimizer) || dense-gradient all-reduce
(sum, like ``hvd.DistributedOptimizer(op=hvd.Sum)`` in the reference benchmark,
test/benchmark/criteo_deepctr.py:262-263) -> dense Adagrad -> D2H(loss).

The whole device part is captured in ONE CUDA graph (launch-bound at batch 4096); the
input copy of step k+1 and the loss read of step k-1 overlap step k.
"""
import torch
import torch.nn.functional as F

from ..context import get_context


class FlatAdagrad:
    """tf.keras Adagrad (lr=0.001, initial_accumulator_value=0.1, eps=1e-7) over ONE flat
    fp32 buffer that aliases every dense parameter -- 3 kernels regardless of the number
    of parameters, graph capturable."""

    def __init__(self, params, lr=0.001, initial_accumulator_value=0.1, eps=1e-7):
        self.params = [p for p in params]
        self.lr, self.eps = lr, eps
        dev = self.params[0].device
        n = sum(p.numel() for p in self.params)
        self.n = n
        self.flat = torch.zeros(n, dtype=torch.float32, device=dev)
        self.grad = torch.zeros(n, dtype=torch.float32, device=dev)
        self.accum = torch.full((n,), initial_accumulator_value, dtype=torch.float32, device=dev)
        off = 0
        for p in self.params:
            k = p.numel()
            self.flat[off:off + k].copy_(p.data.reshape(-1).float())
            p.data = self.flat[off:off + k].view_as(p)
            p.grad = self.grad[off:off + k].view_as(p)
            off += k

    def zero_grad(self):
        self.grad.zero_()

    def step(self):
        g = self.grad
        self.accum.addcmul_(g, g)
        self.flat.addcdiv_(g, self.accum.sqrt().add_(self.eps), value=-self.lr)


class FlatAdam(FlatAdagrad):
    """tf.keras Adam over the flat buffer (the reference benchmark's --optimizer Adam)"""

    def __init__(self, params, lr=0.001, beta_1=0.9, beta_2=0.999, eps=1e-7):
        super().__init__(params, lr=lr, initial_accumulator_value=0.0, eps=eps)
        self.b1, self.b2 = beta_1, beta_2
        self.v = torch.zeros_like(self.accum)
        self.t = torch.zeros((), dtype=torch.float32, device=self.flat.device)

    def step(self):
        g = self.grad
        self.t += 1
        self.accum.mul_(self.b1).add_(g, alpha=1 - self.b1)
        self.v.mul_(self.b2).addcmul_(g, g, value=1 - self.b2)
        lr_t = self.lr * torch.sqrt(1 - self.b2 ** self.t) / (1 - self.b1 ** self.t)
        self.flat.sub_(lr_t * self.accum / (self.v.sqrt() + self.eps))


class FlatFtrl(FlatAdagrad):
    """tf.keras Ftrl over the flat buffer (defaults of the reference benchmark)"""

    def __init__(self, params, lr=0.001, initial_accumulator_value=0.1, l1=0.0, l2=0.0, lr_power=-0.5):
        super().__init__(params, lr=lr, initial_accumulator_value=initial_accumulator_value)
        self.l1, self.l2, self.p = l1, l2, -lr_power
        self.lin = torch.zeros_like(self.accum)

    def step(self):
        g, w = self.grad, self.flat
        an = self.accum + g * g
        sigma = (an.pow(self.p) - self.accum.pow(self.p)) / self.lr
        self.lin.add_(g - sigma * w)
        self.accum.copy_(an)
        quad = an.pow(self.p) / self.lr + 2 * self.l2
        self.flat.copy_((self.lin.clamp(-self.l1, self.l1) - self.lin) / quad)


def make_flat_optimizer(params, config=None, lr=0.001):
    """dense optimizer of the eager trainer from a Keras-style config ({"category": adagrad | adam | ftrl, ...})"""
    from ..config import normalize_optimizer
    c = normalize_optimizer(config or {"category": "adagrad", "learning_rate": lr})
    if c["category"] == "adam":
        return FlatAdam(params, lr=c["learning_rate"], beta_1=c["beta_1"], beta_2=c["beta_2"], eps=c["epsilon"])
    if c["category"] == "ftrl":
        return FlatFtrl(params, lr=c["learning_rate"], initial_accumulator_value=c["initial_accumulator_value"],
                        l1=c["l1_regularization_strength"], l2=c["l2_regularization_strength"], lr_power=c["learning_rate_power"])
    return FlatAdagrad(params, lr=c["learning_rate"], initial_accumulator_value=c.get("initial_accumulator_value", 0.1),
                       eps=c.get("epsilon", 1e-7))


class Trainer:
    def __init__(self, model, lr=0.001, use_graph=True, allreduce="auto", dense_optimizer=None):
        self.ctx = get_context()
        self.model = model
        self.device = self.ctx.device
        self.world = self.ctx.world
        self.opt = make_flat_optimizer(model.dense_parameters(), dense_optimizer, lr=lr)
        self.use_graph = use_graph and self.device.type == "cuda"
        self.graph = None
        self._static = None
        self.allreduce = allreduce
        self._ar = None
        if self.world > 1 and self.device.type == "cuda":
            from ..parallel.allreduce import make_allreduce
            self._ar = make_allreduce(self.ctx, self.opt.grad, mode=allreduce)

    # ---- one device step on given device tensors; returns loss tensor (0-dim, device)
    def _device_step(self, ids, dense, labels):
        from ..utils.timers import nvtx_range
        self.opt.zero_grad()
        with nvtx_range("forward"):
            logits = self.model(ids, dense)
            loss = F.binary_cross_entropy_with_logits(logits, labels)
        with nvtx_range("backward+push_update"):
            loss.backward()
        if self.world > 1:
            if self._ar is not None:
                self._ar()
            else:
                import torch.distributed as dist
                dist.all_reduce(self.opt.grad, group=self.ctx.group)
        self.opt.step()
        return loss.detach()

    def step(self, ids, dense, labels):
        """eager or graph-replayed step on device tensors"""
        if not self.use_graph:
            loss = self._device_step(ids, dense, labels)
            self.ctx.step_done()
            return loss
        if self.graph is None:
            self._capture(ids, dense, labels)
        s = self._static
        if ids.data_ptr() != s["ids"].data_ptr():
            s["ids"].copy_(ids, non_blocking=True)
            s["dense"].copy_(dense, non_blocking=True)
            s["labels"].copy_(labels, non_blocking=True)
        self.graph.replay()
        self.ctx.step_done()
        return s["loss"]

    def _capture(self, ids, dense, labels):
        s = {"ids": ids.clone(), "dense": dense.clone(), "labels": labels.clone()}
        side = torch.cuda.Stream(device=self.device)
        side.wait_stream(torch.cuda.current_stream(self.device))
        with torch.cuda.stream(side):
            # warm-up outside capture (allocator, cuBLAS handles, autotune): PyTorch's whole-network capture recipe --
            # these are three REAL training steps on the first batch (the fused trainer's warm-up is parameter-neutral,
            # FusedCTR.warmup; the autograd-driven eager zoo has no zero-row path through torch's own ops)
            for _ in range(3):
                self._device_step(s["ids"], s["dense"], s["labels"])
        torch.cuda.current_stream(self.device).wait_stream(side)
        torch.cuda.synchronize(self.device)
        if self.world > 1:
            self.ctx.barrier()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            s["loss"] = self._device_step(s["ids"], s["dense"], s["labels"])
        self.graph, self._static = g, s

    def static_inputs(self):
        return self._static

    # ---- end-to-end: pinned host batch in, python float loss out (one step late)
    def make_pipeline(self, batch, num_sparse, num_dense):
        return _Pipeline(self, batch, num_sparse, num_dense)


class _Pipeline:
    """User-facing end-to-end step: ``submit(host_ids, host_dense, host_labels)`` enqueues the H2D copy on a copy
    stream, one training step on the compute stream and an asynchronous D2H of its loss; ``last_loss()`` drains.
    Inputs must be pinned.

    With a trainer that can prefetch (``FusedTrainer``: ``step(..., next_ids=)``) the pipeline runs ONE BATCH
    AHEAD: ``submit(batch k)`` copies batch k and trains batch k-1 with ``next_ids`` = the device ids of batch k,
    so the de-duplication plan of batch k is built while batch k-1 computes -- the reference's ``pulling``
    input-pipeline prefetch (exb.py:645-691). Three device buffers: the copy of batch k+1 overlaps step k-1."""

    NBUF = 3

    def __init__(self, trainer, batch, num_sparse, num_dense):
        self.t = trainer
        dev = trainer.device
        n = self.NBUF
        self.lookahead = bool(getattr(trainer, "supports_prefetch", False)) and bool(getattr(trainer, "want_prefetch", False))
        self.copy_stream = torch.cuda.Stream(device=dev)
        self.dev = [dict(ids=torch.zeros((batch, num_sparse), dtype=torch.int64, device=dev),
                         dense=torch.zeros((batch, num_dense), dtype=torch.float32, device=dev),
                         labels=torch.zeros((batch,), dtype=torch.float32, device=dev)) for _ in range(n)]
        self.loss_host = [torch.zeros((), dtype=torch.float32).pin_memory() for _ in range(n)]
        self.copied = [torch.cuda.Event() for _ in range(n)]
        self.done = [torch.cuda.Event() for _ in range(n)]
        self.k = 0            # batches submitted
        self.trained = 0      # batches trained
        self.waited = -1      # last batch whose copy the compute stream waited for in submit()
        self.h2d_bytes = batch * num_sparse * 8 + batch * num_dense * 4 + batch * 4
        self.d2h_bytes = 4

    def _train(self, j, next_ids, copied_waited=False):
        """launch the step of batch j (device buffer j % NBUF)"""
        i = j % self.NBUF
        cur = torch.cuda.current_stream(self.t.device)
        if not copied_waited:
            cur.wait_event(self.copied[i])
        if j >= self.NBUF:
            self.done[i].synchronize()                        # loss_host[i] of batch j - NBUF has landed
        d = self.dev[i]
        if next_ids is not None and getattr(self.t, "supports_stable_inputs", False):
            # this pipeline's device buffers live as long as the pipeline and are refilled in place
            loss = self.t.step(d["ids"], d["dense"], d["labels"], next_ids=next_ids, stable=True)
        elif next_ids is not None:
            loss = self.t.step(d["ids"], d["dense"], d["labels"], next_ids=next_ids)
        else:
            loss = self.t.step(d["ids"], d["dense"], d["labels"])
        self.loss_host[i].copy_(loss, non_blocking=True)
        self.done[i].record(cur)      # one event: the loss has landed AND buffer i may be refilled (the copy stream waits on it)
        self.trained = j + 1

    def submit(self, ids_h, dense_h, labels_h):
        k = self.k
        i = k % self.NBUF
        if k >= self.NBUF:
            self.copy_stream.wait_event(self.done[i])         # buffer i free again (batch k - NBUF trained)
        with torch.cuda.stream(self.copy_stream):
            d = self.dev[i]
            d["ids"].copy_(ids_h, non_blocking=True)
            d["dense"].copy_(dense_h, non_blocking=True)
            d["labels"].copy_(labels_h, non_blocking=True)
            self.copied[i].record(self.copy_stream)
        self.k = k + 1
        if not self.lookahead:
            self._train(k, None)
        elif self.trained < k:        # right after flush() batch k-1 is trained already; the next submit trains batch k
            cur = torch.cuda.current_stream(self.t.device)
            cur.wait_event(self.copied[i])                    # the plan kernel of batch k reads its ids
            # batch k-1's copy was waited for by the previous submit (as "next ids") -- if that one trained a batch
            self._train(k - 1, self.dev[i]["ids"], copied_waited=self.waited == k - 1)
            self.waited = k

    def flush(self):
        while self.trained < self.k:
            self._train(self.trained, None)

    def last_loss(self):
        self.flush()
        i = (self.k - 1) % self.NBUF
        self.done[i].synchronize()
        return float(self.loss_host[i])
