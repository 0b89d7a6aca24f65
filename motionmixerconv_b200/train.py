"""The training step as one replayable unit: forward -> MPJPE -> backward -> (all-reduce) -> Adam.

``TrainStep`` is the fast path for the loop body of ``h36m/train_mixer_h36m.py:110-195``
(``zero_grad; pred = model(x); loss = mpjpe_error(pred, gt); loss.backward(); optimizer.step()``):

* every parameter of the model becomes a view into ONE flat fp32 buffer, gradients / Adam moments
  live in matching flat buffers (``state_dict`` is unaffected: the nn.Parameters keep their names
  and shapes, only their storage moves);
* the kernels are called straight through the C ABI on preallocated activations — no autograd
  graph, no per-op allocation — and the whole step is captured in a CUDA graph;
* data parallelism: one process per GPU, the batch is sharded by the caller, and ONE
  ``all_reduce(SUM)`` over the flat gradient bucket (NCCL over NVLink) sits between backward and
  the fused Adam, which folds the ``1/world_size`` in.  Replicated optimizer state.

The autograd path (``model(x)`` + any torch optimizer) stays available and produces the same numbers.
"""
from __future__ import annotations

import ctypes as C
import math
import os
import sys

import torch
import torch.distributed as dist

from . import _lib as L
from . import functional as F_
from . import parallel as P_
from .functional import _p


class FlatBuffers:
    """Flat param / grad / exp_avg / exp_avg_sq buffers; parameters are re-pointed to views."""

    def __init__(self, model):
        params = []
        seen = set()
        for p in model.parameters():
            if id(p) not in seen and p.requires_grad:
                seen.add(id(p))
                params.append(p)
        if not params:
            raise ValueError("model has no trainable parameters")
        dev = params[0].device
        if dev.type != "cuda":
            raise RuntimeError("TrainStep needs the model on a CUDA device (model.to('cuda') first)")
        self.params = params
        self.offsets, o = P_.flat_offsets([p.numel() for p in params])   # every view 16-byte aligned
        self.numel = o
        self.p = torch.zeros(o, dtype=torch.float32, device=dev)
        self.g = torch.zeros_like(self.p)
        self.m = torch.zeros_like(self.p)
        self.v = torch.zeros_like(self.p)
        self.grad_views = {}
        with torch.no_grad():
            for p, off in zip(params, self.offsets):
                view = self.p[off:off + p.numel()].view(p.shape)
                view.copy_(p.data)
                p.data = view
        self.rebind_grads(self.g)

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


class _MlpMixerPlan:
    """Pointer tables + static activations for one (model, batch size)."""

    def __init__(self, model, flat, B, dropout_step_dev):
        from .mlp_mixer import MlpMixer
        assert isinstance(model, MlpMixer)
        self.model, self.B = model, B
        dev = flat.p.device
        T, H, D, To = model.seq_len, model.hidden_dim, model.input_size, model.pred_len
        self.x = torch.zeros(B, T, D, device=dev)
        self.acts = [torch.empty(B, T, H, device=dev) for _ in range(model.num_blocks + 1)]
        self.pred = torch.empty(B, To, model.num_classes, device=dev)
        self.dpred = torch.empty_like(self.pred)
        self.dact = [torch.empty(B, T, H, device=dev) for _ in range(2)]
        self.step_dev = dropout_step_dev
        self.blocks = []
        self.bn_runs = {}                 # block index -> (MlpBnBlock, params, grads, bn modules, bn grads): regularization == -1
        for i, mb in enumerate(model.Mixer_Block):
            kp = mb.kernel_params()
            self.blocks.append((mb, F_.mlp_block_table(kp), F_.mlp_block_table([flat.grad_of(q) for q in kp])))
            if mb.regularization == -1.0:     # BatchNorm1d inside the MLP blocks: a chain of stage kernels with static buffers
                bns = mb.bn_modules()
                self.bn_runs[i] = (F_.MlpBnBlock(B, T, H, mb.tokens_mlp_dim, mb.channels_mlp_dim, dev), kp, [flat.grad_of(q) for q in kp],
                                   bns, [(flat.grad_of(m.weight), flat.grad_of(m.bias)) for m in bns])
        hp = [model.LN.weight, model.LN.bias, model.conv_out.weight, model.conv_out.bias, model.fc_out.weight, model.fc_out.bias]
        self.head_w = F_.mlp_head_table(hp)
        self.head_g = F_.mlp_head_table([flat.grad_of(q) for q in hp])
        self.head_desc = L.MmxMlpHeadDesc(B, T, To, H, model.num_classes)
        self.conv_w, self.conv_b = model.conv.weight, model.conv.bias
        self.conv_gw, self.conv_gb = flat.grad_of(model.conv.weight), flat.grad_of(model.conv.bias)
        self.seed = torch.initial_seed() & 0xFFFFFFFFFFFFFFFF
        self.n_launches_fwd = 2 + model.num_blocks
        self.n_launches_bwd = 2 + model.num_blocks
        # kernels that can save the token-half output x1 (+ SE gates) for the backward (the tcgen05 family): one extra tile per block
        lib = L.load()
        self.saves = [i not in self.bn_runs and bool(lib.mmx_mlp_block_saves(C.byref(self._desc(mb, True)))) for i, (mb, _, _) in enumerate(self.blocks)]
        self.x1 = [torch.empty(B, T, H, device=dev) if s else None for s in self.saves]
        self.gate = [torch.empty(B, T, device=dev) if s else None for s in self.saves]
        nb = len(self.bn_runs)
        self.n_launches_fwd = 2 + sum(2 if s else 1 for s in self.saves) - nb + nb * F_.MlpBnBlock.n_launches_fwd   # tcgen05 family: token half + channel half
        self.n_launches_bwd = 2 + sum(2 if s else 1 for s in self.saves) - nb + nb * F_.MlpBnBlock.n_launches_bwd

    def _desc(self, mb, training):
        m = mb.meta(self.seed, 0)
        T, H = self.model.seq_len, self.model.hidden_dim
        return F_.mlp_block_desc(self.B, T, H, *m[:6], training, *m[7:], step_dev=_p(self.step_dev) if training else None)

    def forward(self, lib, st, training):
        md = self.model
        T, H, D = md.seq_len, md.hidden_dim, md.input_size
        prec = L.MMX_PREC[md.precision or F_.get_precision()]
        L.check(lib, lib.mmx_linear_fwd_prec(self.B * T, D, H, _p(self.x), _p(self.conv_w), _p(self.conv_b), _p(self.acts[0]), prec, st), "mmx_linear_fwd")
        for i, (mb, tw, _) in enumerate(self.blocks):
            if i in self.bn_runs:
                run, kp, _, bns, _ = self.bn_runs[i]
                m = mb.meta(0, 0)
                run.forward(self.acts[i], self.acts[i + 1], kp, bns, m[3], m[2] if m[4] else 0, m[5], training)
                continue
            d = self._desc(mb, training)
            if training and self.saves[i]:
                L.check(lib, lib.mmx_mlp_block_fwd_save(C.byref(d), C.byref(tw), _p(self.acts[i]), _p(self.acts[i + 1]), _p(self.x1[i]),
                                                        _p(self.gate[i]), st), "mmx_mlp_block_fwd_save")
            else:
                L.check(lib, lib.mmx_mlp_block_fwd(C.byref(d), C.byref(tw), _p(self.acts[i]), _p(self.acts[i + 1]), st), "mmx_mlp_block_fwd")
        L.check(lib, lib.mmx_mlp_head_fwd_prec(C.byref(self.head_desc), C.byref(self.head_w), _p(self.acts[-1]), _p(self.pred), prec, st), "mmx_mlp_head_fwd")
        return self.pred

    def backward(self, lib, st):
        md = self.model
        T, H, D = md.seq_len, md.hidden_dim, md.input_size
        cur = self.dact[0]
        prec = L.MMX_PREC[md.precision or F_.get_precision()]
        L.check(lib, lib.mmx_mlp_head_bwd_prec(C.byref(self.head_desc), C.byref(self.head_w), C.byref(self.head_g),
                                               _p(self.acts[-1]), _p(self.dpred), _p(cur), prec, st), "mmx_mlp_head_bwd")
        for i in reversed(range(len(self.blocks))):
            mb, tw, tg = self.blocks[i]
            nxt = self.dact[1] if cur is self.dact[0] else self.dact[0]
            if i in self.bn_runs:
                run, kp, kg, _, bg = self.bn_runs[i]
                m = mb.meta(0, 0)
                run.backward(self.acts[i], cur, nxt, kp, kg, bg, m[3], m[2] if m[4] else 0, m[5])
                cur = nxt
                continue
            d = self._desc(mb, True)
            if self.saves[i]:
                L.check(lib, lib.mmx_mlp_block_bwd_saved(C.byref(d), C.byref(tw), C.byref(tg), _p(self.acts[i]), _p(self.x1[i]), _p(self.gate[i]),
                                                         _p(cur), _p(nxt), st), "mmx_mlp_block_bwd_saved")
            else:
                L.check(lib, lib.mmx_mlp_block_bwd(C.byref(d), C.byref(tw), C.byref(tg), _p(self.acts[i]), _p(cur), _p(nxt), st), "mmx_mlp_block_bwd")
            cur = nxt
        L.check(lib, lib.mmx_linear_bwd_prec(self.B * T, D, H, _p(self.x), _p(self.conv_w), _p(cur), _p(self.conv_gw), _p(self.conv_gb), None, prec, st), "mmx_linear_bwd")


class _ConvMixerPlan:
    """Pointer tables + static activations for one (ConvMixer, batch size)."""

    def __init__(self, model, flat, B, dropout_step_dev):
        from .conv_mixer_model import ConvMixer
        assert isinstance(model, ConvMixer)
        self.model, self.B = model, B
        dev = flat.p.device
        T, D, E, C = model.in_nTP, model.dimPosIn, model.dimPosEmb, model.conv_nChan
        To, Dout = model.out_nTP, model.dimPosOut
        enc = model.encoder
        self.Hn = max(int(enc.n_harmonic_functions), 0)
        self.x = torch.zeros(B, T, D, device=dev)
        self.m = torch.empty(B * T, E, device=dev)
        self.dm = torch.empty(B * T, E, device=dev)
        self.step_dev = dropout_step_dev
        self.seed = torch.initial_seed() & 0xFFFFFFFFFFFFFFFF
        ep = [enc.frequencies if self.Hn > 0 else None, enc.embed_mlp.weight, enc.embed_mlp.bias,
              enc.channelUpscaling.weight, enc.channelUpscaling.bias]
        self.enc_w = F_.encoder_table(ep)
        self.enc_g = F_.encoder_table([None] + [flat.grad_of(q) for q in ep[1:]])
        self.enc_desc = L.MmxEncoderDesc(B, T, D, E, C, self.Hn)
        # ops in execution order: ("half", block, half, params table, grads table) | ("tail", block, se ptrs)
        self.ops = []
        self.bn = {}                      # op index -> BatchNorm state of that half (regularization == -1)
        self.large = {}                   # op index -> stage-kernel chain of a half the fused kernels do not serve
        for mb in model.Mixer_Block:
            for half in ((0, 1) if mb.mode_conv == "twice" else (0,)):
                hp = mb.half_params(half)
                if mb.uses_large_path(half, B):
                    reg = (mb.conv1 if half == 0 else mb.conv2).reg if mb.regularization == -1.0 else None
                    self.large[len(self.ops)] = dict(
                        run=F_.ConvHalfLarge(B, C, T, E, dev, with_bn=reg is not None, precision=mb.precision), params=hp, grads=[flat.grad_of(q) for q in hp],
                        reg=reg, bn_grads=None if reg is None else [flat.grad_of(reg.weight), flat.grad_of(reg.bias)])
                elif mb.regularization == -1.0:
                    reg = (mb.conv1 if half == 0 else mb.conv2).reg
                    self.bn[len(self.ops)] = dict(
                        reg=reg, z=torch.empty(B, C, T, E, device=dev), gd=torch.empty(B, T, 2, device=dev),
                        sums=torch.zeros(2 * C, dtype=torch.float64, device=dev), bn=torch.zeros(4 * C, device=dev),
                        coef=torch.zeros(3 * C, device=dev), gw=flat.grad_of(reg.weight), gb=flat.grad_of(reg.bias))
                self.ops.append(("half", mb, half, F_.conv_half_table(hp), F_.conv_half_table([flat.grad_of(q) for q in hp])))
            if mb.mode_conv != "twice":
                s1, s2 = mb.se_weights()
                self.ops.append(("tail", mb, 1, (s1, s2), (flat.grad_of(s1), flat.grad_of(s2))))
        self.acts = [torch.empty(B, C, T, E, device=dev) for _ in range(len(self.ops) + 1)]
        self.pred = torch.empty(B, To, Dout, device=dev)
        self.dpred = torch.empty_like(self.pred)
        self.dact = [torch.empty(B, C, T, E, device=dev) for _ in range(2)]
        hp = model.head_params()
        self.head_w = F_.conv_head_table(hp)
        self.head_g = F_.conv_head_table([flat.grad_of(q) for q in hp])
        self.head_desc = L.MmxConvHeadDesc(B, C, T, To, E, Dout)
        self.n_launches_fwd = 2 + len(self.ops) + sum(F_.ConvHalfLarge.launches(v["reg"] is not None)[0] - 1 for v in self.large.values())
        self.n_launches_bwd = (1 + len(self.ops) + (2 if self.Hn == 0 else 3)
                               + sum(F_.ConvHalfLarge.launches(v["reg"] is not None)[1] - 1 for v in self.large.values()))

    def _desc(self, mb, half, training):
        m = mb.half_meta(half, self.seed, 0)
        md = self.model
        return F_.conv_half_desc(self.B, md.conv_nChan, md.in_nTP, md.dimPosEmb, *m[:6], training, *m[7:],
                                 step_dev=_p(self.step_dev) if training else None)

    def _tail(self, lib, fn, mb, st, *ptrs):
        md = self.model
        return getattr(lib, fn)(self.B, md.conv_nChan, md.in_nTP, md.dimPosEmb, md.in_nTP // mb.r_se if mb.use_se else 0,
                                int(mb.use_se), int(mb.use_max_pooling), *ptrs, st)

    def forward(self, lib, st, training):
        L.check(lib, lib.mmx_pose_encoder_fwd(C.byref(self.enc_desc), C.byref(self.enc_w), _p(self.x), _p(self.m), _p(self.acts[0]), st),
                "mmx_pose_encoder_fwd")
        for i, (kind, mb, half, tw, _) in enumerate(self.ops):
            if kind == "half" and i in self.large:
                lg = self.large[i]
                lg["run"].forward(self._desc(mb, half, training), self.acts[i], self.acts[i + 1], lg["params"], lg["reg"])
            elif kind == "half" and i in self.bn:
                b = self.bn[i]
                d = self._desc(mb, half, training)
                if training:
                    reg = b["reg"]
                    F_.bn_forward_passes(d, tw, self.acts[i], b["z"], self.acts[i + 1], b["sums"], b["bn"], reg.weight, reg.bias,
                                         reg.running_mean, reg.running_var, reg.num_batches_tracked)
                else:
                    aff = F_.bn_eval_affine(b["reg"])
                    hp = mb.half_params(half)
                    L.check(lib, lib.mmx_conv_half_fwd(C.byref(d), C.byref(F_.conv_half_table(hp, aff)), _p(self.acts[i]), _p(self.acts[i + 1]), st),
                            "mmx_conv_half_fwd")
                    self._keep = aff
            elif kind == "half":
                d = self._desc(mb, half, training)
                L.check(lib, lib.mmx_conv_half_fwd(C.byref(d), C.byref(tw), _p(self.acts[i]), _p(self.acts[i + 1]), st), "mmx_conv_half_fwd")
            else:
                L.check(lib, self._tail(lib, "mmx_se_tail_fwd", mb, st, _p(tw[0]), _p(tw[1]), _p(self.acts[i]), _p(self.acts[i + 1])), "mmx_se_tail_fwd")
        L.check(lib, lib.mmx_conv_head_fwd(C.byref(self.head_desc), C.byref(self.head_w), _p(self.acts[-1]), _p(self.pred), st), "mmx_conv_head_fwd")
        return self.pred

    def backward(self, lib, st):
        cur = self.dact[0]
        L.check(lib, lib.mmx_conv_head_bwd(C.byref(self.head_desc), C.byref(self.head_w), C.byref(self.head_g),
                                           _p(self.acts[-1]), _p(self.dpred), _p(cur), st), "mmx_conv_head_bwd")
        for i in reversed(range(len(self.ops))):
            kind, mb, half, tw, tg = self.ops[i]
            nxt = self.dact[1] if cur is self.dact[0] else self.dact[0]
            if kind == "half" and i in self.large:
                lg = self.large[i]
                lg["run"].backward(self._desc(mb, half, True), self.acts[i], cur, nxt, lg["params"], lg["grads"], lg["bn_grads"])
            elif kind == "half" and i in self.bn:
                b = self.bn[i]
                d = self._desc(mb, half, True)
                Bn, Cn, Tn, En = self.acts[i].shape
                F_.bn_backward_passes(d, tw, tg, self.acts[i], b["z"], cur, nxt, b["bn"], b["gd"], b["sums"], b["coef"], b["gw"], b["gb"],
                                      Bn * Tn * En)
            elif kind == "half":
                d = self._desc(mb, half, True)
                L.check(lib, lib.mmx_conv_half_bwd(C.byref(d), C.byref(tw), C.byref(tg), _p(self.acts[i]), _p(cur), _p(nxt), st), "mmx_conv_half_bwd")
            else:
                L.check(lib, self._tail(lib, "mmx_se_tail_bwd", mb, st, _p(tw[0]), _p(tw[1]), _p(tg[0]), _p(tg[1]),
                                        _p(self.acts[i]), _p(cur), _p(nxt)), "mmx_se_tail_bwd")
            cur = nxt
        L.check(lib, lib.mmx_pose_encoder_bwd(C.byref(self.enc_desc), C.byref(self.enc_w), C.byref(self.enc_g), _p(self.x), _p(self.m),
                                              _p(cur), _p(self.dm), None, st), "mmx_pose_encoder_bwd")


def _make_plan(model, flat, B, step_dev, rank=0):
    from .mlp_mixer import MlpMixer
    from .conv_mixer_model import ConvMixer
    if isinstance(model, MlpMixer):
        plan = _MlpMixerPlan(model, flat, B, step_dev)
    elif isinstance(model, ConvMixer):
        plan = _ConvMixerPlan(model, flat, B, step_dev)
    else:
        raise TypeError("TrainStep supports motionmixerconv_b200 MlpMixer / ConvMixer, got %s" % type(model).__name__)
    # data parallel: every rank draws its own dropout masks (identical seeds would give every shard the same masks)
    plan.seed = (plan.seed + 0x9E3779B97F4A7C15 * rank) & 0xFFFFFFFFFFFFFFFF
    return plan


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
        self.flat = FlatBuffers(model)
        self.lr, self.wd, self.betas, self.eps = lr, weight_decay, betas, eps
        self.loss_scale = loss_scale
        self.pg = process_group
        self.world = dist.get_world_size(process_group) if process_group is not None else 1
        self.use_graph = use_cuda_graph
        dev = self.flat.p.device
        self.device = dev
        # optimiser clock and hyper-parameters live on the device (mmx_adam_advance): nothing is
        # written from the host per step, so the step is replayable from a CUDA graph
        self.hyper = torch.tensor([lr, betas[0], betas[1], eps, weight_decay, 1.0, 1.0, 1.0 / self.world, 1 - betas[0], 1 - betas[1]],
                                  dtype=torch.float32, device=dev)
        self.step_dev = torch.zeros(1, dtype=torch.int32, device=dev)
        self.loss_sum = torch.zeros(1, dtype=torch.float32, device=dev)
        self.plan = None
        self.gt = None
        self.graph_a = self.graph_b = None
        self._plans = {}              # batch size -> (plan, gt, graph_a, graph_b): train / eval at different batch sizes do not evict each other
        self.kernel_launches_per_step = 0
        self.rank = dist.get_rank(process_group) if process_group is not None else 0
        if self.world > 1:
            # replicas must start identical (what DDP does at construction): rank 0's parameters and buffers win
            src = dist.get_global_rank(process_group, 0)
            dist.broadcast(self.flat.p, src=src, group=process_group)
            for b in model.buffers():
                dist.broadcast(b, src=src, group=process_group)
        # gradient exchange: by default ONE kernel does the all-reduce over NVLink peer memory and the Adam update
        # (mmx_adam_step_peer); MMX_DP_PEER=0, or peers that cannot be mapped, fall back to an NCCL all-reduce + mmx_adam_step
        self.peer = None
        if self.world > 1 and dev.type == "cuda" and os.environ.get("MMX_DP_PEER", "1") != "0":
            try:
                self.peer = P_.PeerGradBucket(self.flat.numel, dev, process_group)
                self.flat.rebind_grads(self.peer.g)
            except Exception as exc:                         # noqa: BLE001 -- any failure here means "use NCCL"
                self.peer = None
                if self.rank == 0:
                    print("TrainStep: peer-memory gradient exchange unavailable (%s); using the NCCL all-reduce" % exc, file=sys.stderr)
        self._staged, self._copy_stream = None, None      # double-buffered host->device prefetch (step(..., prefetch=...))

    # ---- pieces -------------------------------------------------------------------------------
    def _fwd_bwd(self):
        lib, pl = self.lib, self.plan
        st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        self.flat.g.zero_()
        self.loss_sum.zero_()
        pred = pl.forward(lib, st, training=True)
        n_joints = pred.numel() // 3
        L.check(lib, lib.mmx_mpjpe_fwd_bwd(_p(pred), _p(self.gt), _p(pl.dpred), _p(self.loss_sum), n_joints,
                                           float(self.loss_scale), st), "mmx_mpjpe_fwd_bwd")
        pl.backward(lib, st)

    def _adam(self):
        st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        f = self.flat
        L.check(self.lib, self.lib.mmx_adam_advance(_p(self.hyper), _p(self.step_dev), st), "mmx_adam_advance")
        if self.peer is not None:      # all-reduce over peer memory + Adam, one kernel (collective across the ranks)
            self.peer.adam_step(f.p, f.m, f.v, self.hyper, st)
        else:
            L.check(self.lib, self.lib.mmx_adam_step(_p(f.p), _p(f.g), _p(f.m), _p(f.v), f.numel, _p(self.hyper), st), "mmx_adam_step")

    def _exchange(self):
        """NCCL path only: the peer kernel does the exchange inside _adam."""
        if self.world > 1 and self.peer is None:
            P_.allreduce_bucket(self.flat.g, self.pg)

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
        if lr != self.lr:
            self.lr = lr
            self.hyper[0:1].fill_(lr)

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
            st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
            return self.plan.forward(self.lib, st, training=False)


class FusedAdam(torch.optim.Optimizer):
    """``torch.optim.Adam`` (coupled L2, no amsgrad) as ONE multi-tensor kernel over flat buffers.

    Drop-in for ``optim.Adam(model.parameters(), lr=..., weight_decay=1e-05)``
    (train_mixer_h36m.py:63): ``lr`` is read from ``param_groups`` at every step, so
    ``MultiStepLR`` (:65-67) keeps working.  Parameters are re-pointed to views of a flat buffer on
    the first step; gradients produced by autograd are gathered into the flat gradient buffer.
    """

    def __init__(self, params, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0, process_group=None):
        """``process_group``: batch-sharded data parallelism (one process per GPU): rank 0's parameters are broadcast at the
        first step, every step SUMs the flat gradient bucket over the group and applies 1 / world -- by default inside the
        Adam kernel over NVLink peer memory (mmx_adam_step_peer), else (MMX_DP_PEER=0, peers not mappable) an NCCL all-reduce."""
        super().__init__(params, dict(lr=lr, betas=betas, eps=eps, weight_decay=weight_decay))
        self._flat = {}
        self.pg = process_group
        self.world = dist.get_world_size(process_group) if process_group is not None else 1

    def _flatten(self, gi, group):
        ps = [p for p in group["params"] if p.requires_grad]
        dev = ps[0].device
        if dev.type != "cuda":
            raise RuntimeError("FusedAdam needs CUDA parameters")
        offs, o = [], 0
        for p in ps:
            offs.append(o)
            o += (p.numel() + 3) // 4 * 4
        flat = torch.zeros(o, dtype=torch.float32, device=dev)
        with torch.no_grad():
            for p, off in zip(ps, offs):
                v = flat[off:off + p.numel()].view(p.shape)
                v.copy_(p.data)
                p.data = v
        st = dict(ps=ps, offs=offs, p=flat, g=torch.zeros_like(flat), m=torch.zeros_like(flat), v=torch.zeros_like(flat),
                  hyper=torch.tensor([group["lr"], group["betas"][0], group["betas"][1], group["eps"], group["weight_decay"], 1.0, 1.0, 1.0,
                                      1 - group["betas"][0], 1 - group["betas"][1]],
                                     dtype=torch.float32, device=dev),
                  step=torch.zeros(1, dtype=torch.int32, device=dev), lr=group["lr"], peer=None)
        if self.world > 1:
            st["hyper"][7:8].fill_(1.0 / self.world)
            dist.broadcast(flat, src=dist.get_global_rank(self.pg, 0), group=self.pg)      # replicas start identical
            if os.environ.get("MMX_DP_PEER", "1") != "0":
                try:
                    st["peer"] = P_.PeerGradBucket(o, dev, self.pg)
                    st["g"] = st["peer"].g
                except Exception as exc:                     # noqa: BLE001 -- any failure here means "use NCCL"
                    st["peer"] = None
                    if dist.get_rank(self.pg) == 0:
                        print("FusedAdam: peer-memory gradient exchange unavailable (%s); using the NCCL all-reduce" % exc, file=sys.stderr)
        self._flat[gi] = st
        return st

    @torch.no_grad()
    def step(self, closure=None):
        loss = None
        if closure is not None:
            with torch.enable_grad():
                loss = closure()
        lib = L.load()
        for gi, group in enumerate(self.param_groups):
            st = self._flat.get(gi) or self._flatten(gi, group)
            for p, off in zip(st["ps"], st["offs"]):
                gv = st["g"][off:off + p.numel()]
                if p.grad is None:
                    gv.zero_()
                else:
                    gv.copy_(p.grad.reshape(-1))
            if group["lr"] != st["lr"]:
                st["lr"] = group["lr"]
                st["hyper"][0:1].fill_(group["lr"])
            with torch.cuda.device(st["p"].device):
                stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
                L.check(lib, lib.mmx_adam_advance(_p(st["hyper"]), _p(st["step"]), stream), "mmx_adam_advance")
                if st["peer"] is not None:                   # all-reduce over peer memory + Adam, one kernel (collective)
                    st["peer"].adam_step(st["p"], st["m"], st["v"], st["hyper"], stream)
                else:
                    if self.world > 1:
                        dist.all_reduce(st["g"], op=dist.ReduceOp.SUM, group=self.pg)
                    L.check(lib, lib.mmx_adam_step(_p(st["p"]), _p(st["g"]), _p(st["m"]), _p(st["v"]), st["p"].numel(),
                                                   _p(st["hyper"]), stream), "mmx_adam_step")
        return loss
