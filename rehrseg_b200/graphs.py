"""CUDA-graph replay of a fixed-shape inference forward.

The sliding-window driver (utils/seg_utils.py:267-276) calls the network 8 x (number of tiles) times on identically shaped
tiles; each forward is ~150 short kernel launches, so at B200 speeds the Python / launch overhead, not the GPU, bounds the
loop.  All engine kernels are stream-ordered, allocation-free and take their tensor maps by value, so one forward can be
captured once and replayed with new input contents.
"""
from __future__ import annotations

import weakref

import torch

_graph_cache: "weakref.WeakKeyDictionary" = weakref.WeakKeyDictionary()  # module -> {(shape, dtype): (signature, GraphedForward)}


class GraphedForward:
    """`g = GraphedForward(module, example)`; `g(x)` copies x into the static input, replays the captured forward and
    returns the STATIC output tensors (valid until the next call -- consume or copy them first).

    `range_check=True` captures the forward inside a `rangecheck.RangeCheck(module)`: the graph starts with a memset that zeroes
    its slots, so after each replay `g.range_report()` lists the fp16 saturation of that replay alone (no host synchronisation
    until the report is asked for)."""

    def __init__(self, module, example: torch.Tensor, warmup: int = 2, range_check: bool = False):
        if not example.is_cuda:
            raise ValueError("GraphedForward needs a CUDA example input")
        from . import functional as Fn
        self.static_in = example.detach().clone()
        side = torch.cuda.Stream(device=example.device)
        side.wait_stream(torch.cuda.current_stream(example.device))
        with torch.cuda.stream(side), torch.no_grad():
            for _ in range(warmup):  # packs weights, sets kernel attributes, warms the allocator -- all outside the capture
                module(self.static_in)
        torch.cuda.current_stream(example.device).wait_stream(side)
        torch.cuda.synchronize(example.device)
        self.graph = torch.cuda.CUDAGraph()
        self.range = None
        if range_check:
            from .rangecheck import RangeCheck
            self.range = RangeCheck(module, device=example.device)
        with torch.no_grad(), torch.cuda.graph(self.graph):
            if self.range is None:
                self.static_out = module(self.static_in)
            else:
                self.range.reset()
                with self.range:
                    self.static_out = module(self.static_in)
        # The captured kernels bake in the addresses of the packed 16-bit weight copies made during the warm-up.  Their only
        # other owner is functional's weight cache, which anyone may clear (GraphedTrainStep, bench.py): hold them here so a
        # replay can never read freed memory.  (The module itself is NOT kept: graphed() keys its cache on it weakly.)
        self._packed_weights = [v[2] for v in Fn._wcache.values()]

    def __call__(self, x: torch.Tensor):
        if x.shape != self.static_in.shape:
            raise ValueError(f"GraphedForward captured {tuple(self.static_in.shape)}, got {tuple(x.shape)}")
        self.static_in.copy_(x)
        self.graph.replay()
        return self.static_out

    def range_report(self):
        """fp16 saturation records of the last replay (rangecheck.RangeCheck.report); needs range_check=True."""
        if self.range is None:
            raise ValueError("GraphedForward was captured without range_check=True")
        return self.range.report()


def graphed(module, example: torch.Tensor, range_check: bool = False) -> GraphedForward:
    """Cached GraphedForward for (module, input shape).  The capture bakes in the packed bf16 copies of the weights, so it is
    reused only while every parameter still has the version and storage it had at capture time (an optimiser step or a
    load_state_dict invalidates it)."""
    params = list(module.parameters())
    shape_key = (tuple(example.shape), example.dtype) + (("range_check",) if range_check else ())
    sig = (tuple(p._version for p in params), tuple(p.data_ptr() for p in params))
    per_module = _graph_cache.get(module)
    if per_module is None:
        per_module = _graph_cache[module] = {}   # kept outside the module so state_dict / pickling of the model are unaffected
    hit = per_module.get(shape_key)
    if hit is not None and hit[0] == sig:
        return hit[1]
    for k in [k for k, v in per_module.items() if v[0] != sig]:
        del per_module[k]                         # captures of older weights (any shape) are dead: release their memory
    g = GraphedForward(module, example, range_check=range_check)
    per_module[shape_key] = (sig, g)              # one capture per input shape (single tiles, pairs of mirror variants, ...)
    return g


class GraphedTrainStep:
    """Forward + loss + backward of a fixed-shape training step captured into ONE CUDA graph and replayed.

    A PlainConvUNet step is ~360 kernel launches of 5-400 us; issued from Python the launch latency of the small bottleneck
    layers is exposed (15.06 ms eager vs 14.20 ms replayed for the 2x1x128^3 step on one B200).  Everything the engine does
    is stream-ordered and allocation-free (tensor maps travel by value, workspaces come from PyTorch's caching allocator, no
    host synchronisation), so the whole step -- including the bf16 re-pack of every weight, which reads the CURRENT parameter
    values on every replay -- captures cleanly.

        step = GraphedTrainStep(model, loss_fn, (x, target))      # loss_fn(model(x), target) -> scalar
        for x, target in loader:
            loss = step(x, target)          # copies the batch into the static inputs (host or device source), replays
            opt.step()                      # parameters are updated in place; the .grad tensors are static, overwritten by
                                            # every replay and re-attached to the parameters after it

    The first input is the network input; all inputs must keep their shapes.  `loss` is a static tensor, valid until the next call.

    Data parallel (`dp_group` = a torch.distributed group, or True for the default group): the gradient mean is part of the captured
    step and OVERLAPS the backward pass -- the parameters are cut into `dp_buckets` buckets of equal bytes in the order their
    gradients become final, and as soon as the last gradient of a bucket has been written the bucket is all-reduced (AVG, one
    coalesced NCCL launch over the gradients themselves: no gather / scatter copies) on a communication stream that the compute
    stream joins after the backward pass.  Every rank issues the same collectives in the same (autograd) order.

    `range_check=True`: the step is captured inside a `rangecheck.RangeCheck(model)` whose slots a memset at the start of the
    graph zeroes; `step.range_report()` then lists the fp16 saturation of the last replay's forward pass.
    """

    def __init__(self, model, loss_fn, example_inputs, warmup: int = 2, before_step=None, dp_group=None, dp_buckets: int = 6,
                 range_check: bool = False):
        self.model, self.loss_fn, self.before_step = model, loss_fn, before_step
        self._dp = None
        if dp_group is not None and dp_group is not False:
            import torch.distributed as dist
            if dist.is_available() and dist.is_initialized():
                group = None if dp_group is True else dp_group
                if dist.get_world_size(group) > 1:
                    self._dp = {"group": group, "buckets": int(dp_buckets), "plan": None, "hooks": []}
        self.static_inputs = tuple(t.detach().clone() if t.is_cuda else t.detach().to(next(model.parameters()).device)
                                   for t in example_inputs)
        dev = self.static_inputs[0].device
        self.params = list(model.parameters())
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            if self._dp is not None:
                self._plan_buckets(dev)
            for _ in range(warmup):
                self._eager()
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize(dev)
        for p in self.params:
            p.grad = None                    # gradients are (re)created inside the capture: static addresses, plain assignment
        self.graph = torch.cuda.CUDAGraph()
        # The capture stream has HIGH priority (kernel nodes keep it): the step's main chain and its weight-gradient branch run
        # ahead of the low-priority re-pack branch (functional.SIDE_PRIORITY).
        # thread_local: the NCCL watchdog thread of torch.distributed polls events while this thread captures
        from . import functional as Fn
        cap = torch.cuda.Stream(device=dev, priority=Fn.SIDE_PRIORITY)
        self.range = None
        if range_check:
            from .rangecheck import RangeCheck
            self.range = RangeCheck(model, device=dev)
        l0 = Fn.launches()
        with torch.cuda.graph(self.graph, stream=cap, capture_error_mode="thread_local" if self._dp is not None else "global"):
            if self.range is None:
                self.loss = self._eager()
            else:
                self.range.reset()
                with self.range:
                    self.loss = self._eager()
        self.engine_launches = Fn.launches() - l0      # engine kernels one replay issues (ATen / NCCL nodes not counted)
        self.grads = [p.grad for p in self.params]     # static gradient tensors (None for parameters the loss does not reach)
        # the captured pack kernels write the cached 16-bit weight copies in place: keep them alive with the graph
        from . import functional as Fn
        self._packed_weights = [v[2] for v in Fn._wcache.values()]

    # ---- data-parallel gradient mean, overlapped with the backward pass --------------------------------------------------
    def _plan_buckets(self, dev) -> None:
        """One plain backward with hooks that record the order in which the gradients become final; buckets of equal bytes in
        that order; permanent hooks that fire a bucket's all-reduce when its last gradient has been accumulated."""
        order = []
        hs = [p.register_post_accumulate_grad_hook(lambda q, order=order: order.append(q)) for p in self.params]
        self._plain_step()
        for h in hs:
            h.remove()
        total = sum(p.numel() for p in order)
        nb = max(1, min(self._dp["buckets"], len(order)))
        buckets, cur, acc = [], [], 0
        for p in order:
            cur.append(p)
            acc += p.numel()
            if acc >= total * (len(buckets) + 1) / nb and len(buckets) < nb - 1:
                buckets.append(cur)
                cur = []
        if cur:
            buckets.append(cur)
        self._dp["plan"] = buckets
        self._dp["of"] = {id(p): b for b, ps in enumerate(buckets) for p in ps}
        self._dp["comm"] = torch.cuda.Stream(device=dev)
        self._dp["left"] = [0] * len(buckets)
        self._dp["hooks"] = [p.register_post_accumulate_grad_hook(self._on_grad) for ps in buckets for p in ps]

    def _on_grad(self, p) -> None:
        dp = self._dp
        if not dp.get("armed"):
            return
        b = dp["of"][id(p)]
        dp["left"][b] -= 1
        if dp["left"][b] == 0:
            self._allreduce_bucket(b)

    def _allreduce_bucket(self, b: int) -> None:
        import torch.distributed as dist
        from . import functional as Fn
        dp = self._dp
        dev = self.static_inputs[0].device
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream(dev))
        dp["comm"].wait_event(ev)
        # weight gradients of this bucket may still be running on the side stream: the COMMUNICATION stream waits for them, the
        # compute stream goes on with the backward pass (it joins the side stream at the end of the step)
        ev_side = Fn.pending_wgrad_event()
        if ev_side is not None:
            dp["comm"].wait_event(ev_side)
        with torch.cuda.stream(dp["comm"]):
            with dist._coalescing_manager(group=dp["group"], device=dev, async_ops=False):
                for q in dp["plan"][b]:
                    dist.all_reduce(q.grad, op=dist.ReduceOp.AVG, group=dp["group"])

    def _plain_step(self):
        for p in self.params:
            p.grad = None
        out = self.model(self.static_inputs[0])
        loss = self.loss_fn(out, *self.static_inputs[1:])
        loss.backward()
        return loss

    def _eager(self):
        from . import functional as Fn
        # the 16-bit operand copies must be re-derived INSIDE the captured step from the live parameters (a plain cache hit at
        # capture time would bake stale weights into the graph): every cached copy is re-packed in place on a side stream
        # (a parallel branch of the graph) while the first layers run; the first warm-up step packs lazily instead
        Fn.refresh_weight_cache()
        if self.before_step is not None:
            self.before_step()
        for p in self.params:
            p.grad = None
        out = self.model(self.static_inputs[0])
        loss = self.loss_fn(out, *self.static_inputs[1:])
        if self._dp is not None:
            self._dp["left"] = [len(ps) for ps in self._dp["plan"]]
            self._dp["armed"] = True
        try:
            with Fn.deferred_wgrad():    # this step owns every .grad until it returns: weight gradients join at the end
                loss.backward()
        finally:
            if self._dp is not None:
                self._dp["armed"] = False
        if self._dp is not None:                 # the compute stream continues after every bucket's all-reduce
            dev = self.static_inputs[0].device
            ev = torch.cuda.Event()
            ev.record(self._dp["comm"])
            torch.cuda.current_stream(dev).wait_event(ev)
        Fn._join_prepack()   # (a model without a cached operand copy never joined the pack branch)
        Fn.join_pending_wgrad()
        return loss.detach()

    def close(self) -> None:
        """Drop the captured graph (and the gradient hooks).  REQUIRED before `torch.distributed.destroy_process_group()` when the
        data-parallel all-reduces were captured: tearing the NCCL communicator down while a live graph still holds its kernels
        blocks forever (observed on B200 / torch 2.11 / NCCL 2.28)."""
        if self._dp is not None:
            for h in self._dp.get("hooks", []):
                h.remove()
            self._dp["hooks"] = []
        self.graph = None
        self.grads = None
        dev = self.static_inputs[0].device
        torch.cuda.synchronize(dev)

    def load(self, *inputs, non_blocking: bool = True):
        """Copy a batch (pinned host or device tensors) into the static input buffers on the current stream."""
        for dst, src in zip(self.static_inputs, inputs):
            if src is not dst:
                dst.copy_(src, non_blocking=non_blocking)

    def range_report(self):
        """fp16 saturation records of the last replay (rangecheck.RangeCheck.report); needs range_check=True."""
        if self.range is None:
            raise ValueError("GraphedTrainStep was captured without range_check=True")
        return self.range.report()

    def replay(self):
        self.graph.replay()
        for p, g in zip(self.params, self.grads):      # re-attach the static gradients (zero_grad(set_to_none=True) or an
            p.grad = g                                 # eager step in between may have replaced them)
        return self.loss

    def __call__(self, *inputs):
        self.load(*inputs)
        return self.replay()
