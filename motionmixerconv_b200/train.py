"""The training step as one replayable unit: forward -> MPJPE -> backward -> (all-reduce) -> Adam.

``TrainStep`` is the fast path for the loop body of ``h36m/train_mixer_h36m.py:110-195``
(``zero_grad; pred = model(x); loss = mpjpe_error(pred, gt); loss.backward(); optimizer.step()``):

* every parameter of the model becomes a view into ONE flat fp32 buffer, gradients / Adam moments
  live in matching flat buffers (``state_dict`` is unaffected: the nn.Parameters keep their names
  and shapes, only their storage moves);
* the model's layer runners (``model.runners``, functional.py) — the same kernel sequence as ``model(x)`` — are built once
  per batch size over preallocated activations and the flat gradient bucket, and run without autograd graph or per-op
  allocation; the whole step is captured in a CUDA graph;
* data parallelism: one process per GPU, the batch is sharded by the caller, and ONE
  ``all_reduce(SUM)`` over the flat gradient bucket (NCCL over NVLink) sits between backward and
  the fused Adam, which folds the ``1/world_size`` in.  Replicated optimizer state.

The autograd path (``model(x)`` + any torch optimizer, or ``FusedAdam``, which runs the same flat-buffer Adam update) launches
the same kernels with the same arguments and produces the same numbers.
"""
from __future__ import annotations

import ctypes as C
import os
import sys

import torch
import torch.distributed as dist

from . import _lib as L
from . import functional as F_
from . import parallel as P_
from .functional import _p


class FlatBuffers:
    """Flat param / grad / exp_avg / exp_avg_sq buffers and the on-device Adam state of one parameter list; the parameters are
    re-pointed to views.  ``process_group``: batch-sharded data parallelism.  Rank 0's parameters are broadcast to the group
    (replicas start identical, as DDP does at construction) and the gradient exchange is set up: by default ONE kernel does the
    all-reduce over NVLink peer memory and the Adam update (mmx_adam_step_peer); MMX_DP_PEER=0, or peers that cannot be mapped,
    fall back to an NCCL all-reduce + mmx_adam_step."""

    def __init__(self, params, lr, betas, eps, weight_decay, process_group=None):
        ps, seen = [], set()
        for p in params:
            if id(p) not in seen and p.requires_grad:
                seen.add(id(p))
                ps.append(p)
        if not ps:
            raise ValueError("no trainable parameters")
        dev = ps[0].device
        if dev.type != "cuda":
            raise RuntimeError("the flat parameter buffers need CUDA parameters (model.to('cuda') first)")
        self.params, self.lr = ps, lr
        self.offsets, o = P_.flat_offsets([p.numel() for p in ps])   # every view 16-byte aligned
        self.numel = o
        self.p = torch.zeros(o, dtype=torch.float32, device=dev)
        self.g = torch.zeros_like(self.p)
        self.m = torch.zeros_like(self.p)
        self.v = torch.zeros_like(self.p)
        self.grad_views = {}
        with torch.no_grad():
            for p, off in zip(ps, self.offsets):
                view = self.p[off:off + p.numel()].view(p.shape)
                view.copy_(p.data)
                p.data = view
        self.rebind_grads(self.g)
        self.pg = process_group
        self.world = dist.get_world_size(process_group) if process_group is not None else 1
        # optimiser clock and hyper-parameters live on the device (mmx_adam_advance): nothing is written from the host per
        # step, so the update is replayable from a CUDA graph
        self.hyper = torch.tensor([lr, betas[0], betas[1], eps, weight_decay, 1.0, 1.0, 1.0 / self.world, 1 - betas[0], 1 - betas[1]],
                                  dtype=torch.float32, device=dev)
        self.step = torch.zeros(1, dtype=torch.int32, device=dev)
        self.peer = None
        if self.world > 1:
            dist.broadcast(self.p, src=dist.get_global_rank(process_group, 0), group=process_group)
            if os.environ.get("MMX_DP_PEER", "1") != "0":
                try:
                    self.peer = P_.PeerGradBucket(self.numel, dev, process_group)
                    self.rebind_grads(self.peer.g)
                except Exception as exc:                         # noqa: BLE001 -- any failure here means "use NCCL"
                    self.peer = None
                    if dist.get_rank(process_group) == 0:
                        print("motionmixerconv_b200: peer-memory gradient exchange unavailable (%s); using the NCCL all-reduce" % exc,
                              file=sys.stderr)

    def rebind_grads(self, g):
        """Use ``g`` (flat fp32, same length) as the gradient bucket: e.g. IPC-shared memory for the peer all-reduce."""
        assert g.numel() == self.numel and g.dtype == torch.float32
        self.g = g
        self.grad_views = {id(p): g[off:off + p.numel()].view(p.shape) for p, off in zip(self.params, self.offsets)}

    def grad_of(self, p):
        return None if p is None else self.grad_views[id(p)]

    def attach_grads(self):
        """Expose the flat gradient buffer through ``param.grad`` (for clip_grad_norm_, inspection)."""
        for p in self.params:
            p.grad = self.grad_views[id(p)]

    def set_lr(self, lr):
        if lr != self.lr:
            self.lr = lr
            self.hyper[0:1].fill_(lr)

    def exchange(self):
        """NCCL path only: SUM the gradient bucket over the group (the peer kernel does the exchange inside ``adam``)."""
        if self.world > 1 and self.peer is None:
            P_.allreduce_bucket(self.g, self.pg)

    def adam(self, stream):
        """Advance the optimiser clock, then Adam over the flat buffers: with the peer all-reduce in the same kernel (collective
        across the ranks), else on the (already exchanged) local bucket.  The 1 / world of the mean is hyper[7]."""
        lib = L.load()
        L.check(lib, lib.mmx_adam_advance(_p(self.hyper), _p(self.step), stream), "mmx_adam_advance")
        if self.peer is not None:
            self.peer.adam_step(self.p, self.m, self.v, self.hyper, stream)
        else:
            L.check(lib, lib.mmx_adam_step(_p(self.p), _p(self.g), _p(self.m), _p(self.v), self.numel, _p(self.hyper), stream), "mmx_adam_step")


class _Plan:
    """The model's runners over static activations and the flat gradient bucket, for one (model, batch size): ``x`` -> runs[0]
    -> acts[0] -> runs[1] -> ... -> acts[-1] -> runs[-1] -> ``pred``; the backward ping-pongs over ``dact``."""

    def __init__(self, model, flat, B, step_dev, seed):
        dev = flat.p.device
        self.model, self.B, self.seed = model, B, seed
        self.runs = list(model.runners(B, dev, True, (seed, 0, _p(step_dev))))
        self.grads = [[flat.grad_of(q) for q in r.params] for r in self.runs]
        self.x = torch.zeros(self.runs[0].in_shape, device=dev)
        self.acts = [torch.empty(r.out_shape, device=dev) for r in self.runs[:-1]]
        self.pred = torch.empty(self.runs[-1].out_shape, device=dev)
        self.dpred = torch.empty_like(self.pred)
        self.dact = [torch.empty_like(self.acts[0]) for _ in range(2)]
        self.n_launches_fwd = sum(r.launches[0] for r in self.runs)
        self.n_launches_bwd = sum(r.launches[1] for r in self.runs)

    def forward(self, training):
        for run, x, y in zip(self.runs, [self.x] + self.acts, self.acts + [self.pred]):
            run.forward(x, y, training)
        return self.pred

    def backward(self):
        dy = self.dpred
        for i in reversed(range(len(self.runs))):
            dx = None if i == 0 else (self.dact[1] if dy is self.dact[0] else self.dact[0])
            self.runs[i].backward(self.x if i == 0 else self.acts[i - 1], dy, dx, self.grads[i])
            dy = dx


class _MlpMixerPlan(_Plan):
    """Views for the kernel benchmarks: ``blocks[i] == (block, params table, grads table)``, ``saves`` / ``x1`` / ``gate`` of
    the save variant, and ``_desc(block, training)``; block i reads acts[i]."""

    def __init__(self, *args):
        super().__init__(*args)
        blocks = self.runs[1:-1]
        self.blocks = [(r.mb, F_.mlp_block_table(r.params[:14]), F_.mlp_block_table(g[:14])) for r, g in zip(blocks, self.grads[1:-1])]
        self.saves = [r.saves for r in blocks]
        self.x1 = [r.x1 if r.saves else None for r in blocks]
        self.gate = [r.gate if r.saves else None for r in blocks]

    def _desc(self, mb, training):
        return next(r for r in self.runs if getattr(r, "mb", None) is mb)._desc(training)


class _ConvMixerPlan(_Plan):
    """Views for the kernel benchmarks: ``ops[i] == ("half", block, half, params table, grads table)`` or ``("tail", block, 1,
    SE weights, their gradients)``, ``bn[i]``: the buffers of the fused BatchNorm halves, and ``_desc(block, half, training)``;
    op i reads acts[i]."""

    def __init__(self, *args):
        super().__init__(*args)
        self.ops, self.bn = [], {}
        for i, (r, g) in enumerate(zip(self.runs[1:-1], self.grads[1:-1])):
            if isinstance(r, F_.SeTail):
                self.ops.append(("tail", r.mb, 1, tuple(r.params), tuple(g)))
                continue
            self.ops.append(("half", r.mb, r.half, F_.conv_half_table(r.params[:6]), F_.conv_half_table(g[:6])))
            if isinstance(r, F_.ConvHalf) and r.bnm is not None:
                self.bn[i] = vars(r)

    def _desc(self, mb, half, training):
        return next(r for r in self.runs if getattr(r, "mb", None) is mb and getattr(r, "half", None) == half)._desc(training)


def _make_plan(model, flat, B, step_dev, rank=0):
    from .mlp_mixer import MlpMixer
    from .conv_mixer_model import ConvMixer
    # data parallel: every rank draws its own dropout masks (identical seeds would give every shard the same masks)
    seed = ((torch.initial_seed() & 0xFFFFFFFFFFFFFFFF) + 0x9E3779B97F4A7C15 * rank) & 0xFFFFFFFFFFFFFFFF
    if isinstance(model, MlpMixer):
        return _MlpMixerPlan(model, flat, B, step_dev, seed)
    if isinstance(model, ConvMixer):
        return _ConvMixerPlan(model, flat, B, step_dev, seed)
    raise TypeError("TrainStep supports motionmixerconv_b200 MlpMixer / ConvMixer, got %s" % type(model).__name__)


class TrainStep:
    """``loss = step(x, gt)`` == one iteration of the reference training loop, fused.

    Args mirror the reference call sites: ``lr`` / ``weight_decay`` as in
    ``optim.Adam(model.parameters(), lr=args.lr, weight_decay=1e-05)`` (train_mixer_h36m.py:63);
    ``loss_scale`` is the ``*1000`` of amass/train_mixer_amass.py:92.  ``process_group``: a
    torch.distributed group for batch-sharded data parallelism (None = single GPU).
    """

    def __init__(self, model, lr=1e-3, weight_decay=1e-5, betas=(0.9, 0.999), eps=1e-8, loss_scale=1.0,
                 process_group=None, use_cuda_graph=True):
        self.model = model
        self.lib = L.load()
        self.flat = FlatBuffers(model.parameters(), lr, betas, eps, weight_decay, process_group)
        self.lr, self.wd, self.betas, self.eps = lr, weight_decay, betas, eps
        self.loss_scale = loss_scale
        self.pg = process_group
        self.world = self.flat.world
        self.use_graph = use_cuda_graph
        self.device = self.flat.p.device
        self.hyper, self.step_dev, self.peer = self.flat.hyper, self.flat.step, self.flat.peer
        self.loss_sum = torch.zeros(1, dtype=torch.float32, device=self.device)
        self.plan = None
        self.gt = None
        self.graph_a = self.graph_b = None
        self._plans = {}              # batch size -> (plan, gt, graph_a, graph_b): train / eval at different batch sizes do not evict each other
        self.kernel_launches_per_step = 0
        self.rank = dist.get_rank(process_group) if process_group is not None else 0
        if self.world > 1:            # the model's buffers start identical too (FlatBuffers broadcast the parameters)
            for b in model.buffers():
                dist.broadcast(b, src=dist.get_global_rank(process_group, 0), group=process_group)
        self._staged, self._copy_stream = None, None      # double-buffered host->device prefetch (step(..., prefetch=...))

    # ---- pieces -------------------------------------------------------------------------------
    def _fwd_bwd(self):
        lib, pl = self.lib, self.plan
        st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        self.flat.g.zero_()
        self.loss_sum.zero_()
        pred = pl.forward(training=True)
        n_joints = pred.numel() // 3
        L.check(lib, lib.mmx_mpjpe_fwd_bwd(_p(pred), _p(self.gt), _p(pl.dpred), _p(self.loss_sum), n_joints,
                                           float(self.loss_scale), st), "mmx_mpjpe_fwd_bwd")
        pl.backward()

    def _adam(self):
        self.flat.adam(C.c_void_p(torch.cuda.current_stream().cuda_stream))

    def _exchange(self):
        self.flat.exchange()

    def _select_plan(self, B):
        """Make the plan (static activations, pointer tables, captured graphs) of batch size B current."""
        if self.plan is not None and self.plan.B == B:
            return
        if self.plan is not None:
            self._plans[self.plan.B] = (self.plan, self.gt, self.graph_a, self.graph_b)
        if B in self._plans:
            self.plan, self.gt, self.graph_a, self.graph_b = self._plans[B]
        else:
            self.plan = _make_plan(self.model, self.flat, B, self.step_dev, self.rank)
            self.gt, self.graph_a, self.graph_b = None, None, None
        self.kernel_launches_per_step = self.plan.n_launches_fwd + self.plan.n_launches_bwd + 3  # + mpjpe, adam_advance, adam

    def _prepare(self, x, gt):
        self._select_plan(x.shape[0])
        if tuple(x.shape) != tuple(self.plan.x.shape):
            raise RuntimeError("TrainStep: input %s does not match the model's [B, %d, %d]" % (tuple(x.shape), *self.plan.x.shape[1:]))
        if self.gt is None or tuple(self.gt.shape) != tuple(gt.shape):
            if tuple(gt.shape[1:]) != tuple(self.plan.pred.shape[1:]) or gt.shape[0] != x.shape[0]:
                raise RuntimeError("TrainStep: target %s does not match the prediction %s" % (tuple(gt.shape), tuple(self.plan.pred.shape)))
            self.gt = torch.empty(gt.shape, dtype=torch.float32, device=self.device)
            self.graph_a = self.graph_b = None       # the captured step reads the target buffer

    # ---- optimiser state (the reference never saves it, train_mixer_h36m.py:276; resuming a run needs it) ----
    def _named_flat(self):
        names = {}
        for n, p in self.model.named_parameters():
            names.setdefault(id(p), n)
        return [(names[id(p)], off, p.numel(), p.shape) for p, off in zip(self.flat.params, self.flat.offsets)]

    def state_dict(self):
        """Adam state keyed by parameter name (``exp_avg`` / ``exp_avg_sq`` like torch.optim.Adam) + step count and
        hyper-parameters; pair it with ``model.state_dict()`` in a checkpoint."""
        f = self.flat
        return {"step": self.steps_done, "lr": self.lr, "weight_decay": self.wd, "betas": tuple(self.betas), "eps": self.eps,
                "exp_avg": {n: f.m[o:o + k].view(sh).clone() for n, o, k, sh in self._named_flat()},
                "exp_avg_sq": {n: f.v[o:o + k].view(sh).clone() for n, o, k, sh in self._named_flat()}}

    def load_state_dict(self, sd):
        f = self.flat
        named = self._named_flat()
        missing = [n for n, *_ in named if n not in sd["exp_avg"] or n not in sd["exp_avg_sq"]]
        if missing:
            raise KeyError("TrainStep.load_state_dict: missing optimiser state for %s" % missing)
        with torch.no_grad():
            for n, o, k, sh in named:
                f.m[o:o + k].view(sh).copy_(sd["exp_avg"][n])
                f.v[o:o + k].view(sh).copy_(sd["exp_avg_sq"][n])
            self.step_dev.fill_(int(sd["step"]))
        self.set_lr(float(sd.get("lr", self.lr)))

    def release_graphs(self):
        """Drop every captured CUDA graph (they are re-captured on the next step).  Call before
        ``torch.distributed.destroy_process_group()``: a graph that holds a captured NCCL all-reduce keeps the communicator
        busy and tearing the process group down under it does not return."""
        import gc
        self.graph_a = self.graph_b = None
        self._plans = {B: (pl, gt, None, None) for B, (pl, gt, _, _) in self._plans.items()}
        gc.collect()
        torch.cuda.synchronize(self.device)

    def set_lr(self, lr):
        """Change the learning rate (e.g. from a MultiStepLR schedule, train_mixer_h36m.py:65-67,249)."""
        self.lr = lr
        self.flat.set_lr(lr)

    @property
    def steps_done(self):
        return int(self.step_dev.item())

    # ---- public -------------------------------------------------------------------------------
    def step(self, x, gt, prefetch=None):
        """x: [B,T,D], gt: [B,To,D] (CUDA or pinned host tensors).  Returns the loss as a 0-d CUDA tensor
        (mean MPJPE of THIS rank's shard times ``loss_scale``); no host synchronisation.

        ``prefetch=(x_next, gt_next)`` (pinned host tensors): the NEXT step's inputs start their host->device copy on a side
        stream now, overlapping this step's kernels (what ``DataLoader(pin_memory=True)`` + ``.to(device, non_blocking=True)``
        gives the reference loop, train_mixer_h36m.py:95-96,111).  The next ``step`` call recognises the same tensors and
        only pays a device-to-device copy."""
        if not self.model.training:
            raise RuntimeError("TrainStep.step: the model is in eval() mode (use predict() for inference, model.train() to train)")
        self._prepare(x, gt)
        pl = self.plan
        cur = torch.cuda.current_stream(self.device)
        st = self._staged
        if st is not None and st["x_src"] is x and st["gt_src"] is gt:
            cur.wait_event(st["ready"])
            pl.x.copy_(st["x"], non_blocking=True)
            self.gt.copy_(st["gt"], non_blocking=True)
            st["free"].record(cur)
        else:
            pl.x.copy_(x, non_blocking=True)
            self.gt.copy_(gt, non_blocking=True)
        if prefetch is not None:
            self._prefetch(*prefetch)
        return self._run_step()

    def _prefetch(self, x_next, gt_next):
        if self._copy_stream is None:
            self._copy_stream = torch.cuda.Stream(device=self.device)
        st = self._staged
        if st is None or st["x"].shape != x_next.shape or st["gt"].shape != gt_next.shape:
            st = self._staged = dict(x=torch.empty(x_next.shape, device=self.device), gt=torch.empty(gt_next.shape, device=self.device),
                                     ready=torch.cuda.Event(), free=torch.cuda.Event(), x_src=None, gt_src=None)
            st["free"].record(torch.cuda.current_stream(self.device))
        with torch.cuda.stream(self._copy_stream):
            self._copy_stream.wait_event(st["free"])        # the staging buffers were consumed by the step that used them
            st["x"].copy_(x_next, non_blocking=True)
            st["gt"].copy_(gt_next, non_blocking=True)
            st["ready"].record(self._copy_stream)
        st["x_src"], st["gt_src"] = x_next, gt_next

    def _run_step(self):
        with torch.cuda.device(self.device):
            return self._run_step_on_device()

    def _run_step_on_device(self):
        pl = self.plan
        if not self.use_graph:
            self._fwd_bwd()
            self._exchange()
            self._adam()
        else:
            if self.graph_a is None:
                self._capture()
            self.graph_a.replay()
            if self.graph_b is not None:          # two-graph form (NCCL path): eager all-reduce between backward and Adam
                self._exchange()
                self.graph_b.replay()
        n_joints = pl.pred.numel() // 3
        return (self.loss_sum * (float(self.loss_scale) / n_joints)).reshape(())

    def step_raw(self, batch, dim_used, input_n, output_n, x_scale=1.0, gt_scale=1.0):
        """One training step straight from the raw dataset window (train_mixer_h36m.py:110-120,179): ``batch`` is
        [B, >= input_n+output_n, D_full]; the ``dim_used`` gather, the ``/1000`` and the train / target split run as ONE kernel
        writing into the step's static input buffers (no intermediate tensors)."""
        B = batch.shape[0]
        D = len(dim_used)
        if batch.dim() != 3 or batch.shape[1] < input_n + output_n:
            raise RuntimeError("step_raw: batch %s holds fewer than input_n + output_n = %d frames" % (tuple(batch.shape), input_n + output_n))
        idx = torch.as_tensor(dim_used)
        if idx.numel() and (int(idx.min()) < 0 or int(idx.max()) >= batch.shape[2]):
            raise IndexError("step_raw: dim_used index out of range for a batch with %d dims" % batch.shape[2])
        # shapes are validated against the model by _prepare (static buffers are never written past their end)
        self._prepare(torch.empty(B, input_n, D, device="meta"), torch.empty(B, output_n, D, device="meta"))
        if not isinstance(dim_used, torch.Tensor) or dim_used.device != self.device or dim_used.dtype != torch.int32:
            dim_used = torch.as_tensor(dim_used, dtype=torch.int32).to(self.device)
        F_.window_split(batch.to(self.device, non_blocking=True), dim_used, input_n, output_n, x_scale, gt_scale,
                        out=(self.plan.x, self.gt))
        return self._run_step()

    def _capture(self):
        # warm-up on a side stream (first launches set kernel attributes), then capture
        s = torch.cuda.Stream(device=self.device)
        s.wait_stream(torch.cuda.current_stream())
        state = [self.flat.p, self.flat.m, self.flat.v, self.hyper, self.step_dev, *self.model.buffers()]   # incl. BN running stats
        saved = [b.clone() for b in state]
        with torch.cuda.stream(s):
            self._fwd_bwd()
            self._exchange()                                   # NCCL path: also initialises the communicator before any capture
            self._adam()
        torch.cuda.current_stream().wait_stream(s)
        torch.cuda.synchronize(self.device)
        with torch.no_grad():
            for b, sv in zip(state, saved):
                b.copy_(sv)
        # data parallel: the NCCL all-reduce CAN be captured into the same graph (MMX_DP_GRAPH_ALLREDUCE=1), but measured on
        # 8 x B200 the captured collective has a heavy tail (median step 0.918 ms, mean 1.55 ms) while the eager call between
        # two graphs is steady (0.914 / 0.914 ms): two graphs + eager all-reduce is the default
        one_graph = (self.world == 1 or (self.peer is not None and os.environ.get("MMX_DP_PEER_GRAPHS", "1") != "2")
                     or os.environ.get("MMX_DP_GRAPH_ALLREDUCE", "0") == "1")
        self.graph_a = torch.cuda.CUDAGraph()
        if one_graph:
            # ONE graph per step: forward, backward, the NCCL all-reduce of the flat gradient bucket (NCCL collectives are
            # capturable) and the fused Adam -- no host round trip between backward, the collective and the optimizer
            with torch.cuda.graph(self.graph_a):
                self._fwd_bwd()
                self._exchange()
                self._adam()
            self.graph_b = None
        else:
            with torch.cuda.graph(self.graph_a):
                self._fwd_bwd()
            self.graph_b = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph_b):
                self._adam()

    @torch.no_grad()
    def predict(self, x):
        """Inference forward through the same preallocated plan (eval semantics: no dropout)."""
        self._select_plan(x.shape[0])            # never touches the target buffer / captured graphs of the training plan
        if tuple(x.shape) != tuple(self.plan.x.shape):
            raise RuntimeError("TrainStep.predict: input %s does not match the model's [B, %d, %d]" % (tuple(x.shape), *self.plan.x.shape[1:]))
        with torch.cuda.device(self.device):
            self.plan.x.copy_(x, non_blocking=True)
            return self.plan.forward(training=False)


class FusedAdam(torch.optim.Optimizer):
    """``torch.optim.Adam`` (coupled L2, no amsgrad) as ONE multi-tensor kernel over flat buffers.

    Drop-in for ``optim.Adam(model.parameters(), lr=..., weight_decay=1e-05)``
    (train_mixer_h36m.py:63): ``lr`` is read from ``param_groups`` at every step, so
    ``MultiStepLR`` (:65-67) keeps working.  Each parameter group's parameters are re-pointed to views of a
    ``FlatBuffers`` on the first step; gradients produced by autograd are gathered into its flat gradient buffer.
    """

    def __init__(self, params, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0, process_group=None):
        """``process_group``: batch-sharded data parallelism (one process per GPU): rank 0's parameters are broadcast at the
        first step, every step SUMs the flat gradient bucket over the group and applies 1 / world -- by default inside the
        Adam kernel over NVLink peer memory (mmx_adam_step_peer), else (MMX_DP_PEER=0, peers not mappable) an NCCL all-reduce."""
        super().__init__(params, dict(lr=lr, betas=betas, eps=eps, weight_decay=weight_decay))
        self._flat = {}               # group index -> FlatBuffers
        self.pg = process_group

    def flat(self, gi):
        """The FlatBuffers of parameter group ``gi`` (built, and the parameters re-pointed, on first use)."""
        if gi not in self._flat:
            g = self.param_groups[gi]
            self._flat[gi] = FlatBuffers(g["params"], g["lr"], g["betas"], g["eps"], g["weight_decay"], self.pg)
        return self._flat[gi]

    @torch.no_grad()
    def step(self, closure=None):
        loss = None
        if closure is not None:
            with torch.enable_grad():
                loss = closure()
        for gi, group in enumerate(self.param_groups):
            f = self.flat(gi)
            for p in f.params:
                gv = f.grad_views[id(p)]
                if p.grad is None:
                    gv.zero_()
                else:
                    gv.copy_(p.grad)
            f.set_lr(group["lr"])
            with torch.cuda.device(f.p.device):
                f.exchange()
                f.adam(C.c_void_p(torch.cuda.current_stream().cuda_stream))
        return loss
