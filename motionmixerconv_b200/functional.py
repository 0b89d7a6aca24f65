"""torch.autograd.Function wrappers over the libmmx C ABI (include/mmx.h).

Every op here launches hand-written sm_100a kernels on ``torch.cuda.current_stream()``; inputs must
be CUDA fp32 tensors.  There is no CPU / eager-PyTorch implementation: non-CUDA input raises.
Backward runs on PyTorch's autograd worker thread — the C ABI holds no thread-local CUDA state and
takes the stream explicitly, and we re-enter the tensor's device before every call.
"""
from __future__ import annotations

import ctypes as C
import os
import ctypes as C_   # (the conv wrappers use C for the channel count)

import torch

from . import _lib as L


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _chk(t, name):
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise RuntimeError("motionmixerconv_b200: %s must be a CUDA tensor (the hot path has no CPU implementation)" % name)
    if t.dtype != torch.float32:
        raise RuntimeError("motionmixerconv_b200: %s must be float32, got %s" % (name, t.dtype))
    return t if t.is_contiguous() else t.contiguous()


def _p(t):
    return None if t is None else t.data_ptr()


def _zeros_like_many(tensors):
    """One memset for all gradient buffers: a flat zero buffer sliced into views (16-byte aligned)."""
    sizes = [0 if t is None else (t.numel() + 3) // 4 * 4 for t in tensors]
    ref = next(t for t in tensors if t is not None)
    flat = torch.zeros(sum(sizes), dtype=torch.float32, device=ref.device)
    out, o = [], 0
    for t, n in zip(tensors, sizes):
        out.append(None if t is None else flat[o:o + t.numel()].view(t.shape))
        o += n
    return out


def _call(name, *args):
    lib = L.load()
    L.check(lib, getattr(lib, name)(*args), name)


# ------------------------------------------------------------------------------------------------
# per-frame linear layer (MlpMixer.conv, mlp_mixer.py:325-327)
# ------------------------------------------------------------------------------------------------
class _Linear(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, w, b, precision):
        x, w, b = _chk(x, "x"), _chk(w, "weight"), _chk(b, "bias")
        ctx.prec = L.MMX_PREC[precision or _PRECISION]
        K, N = x.shape[-1], b.numel()
        rows = x.numel() // K
        y = torch.empty(*x.shape[:-1], N, dtype=torch.float32, device=x.device)
        with torch.cuda.device_of(x):
            _call("mmx_linear_fwd_prec", rows, K, N, _p(x), _p(w), _p(b), _p(y), ctx.prec, _stream())
        ctx.save_for_backward(x, w)
        ctx.need_dx = ctx.needs_input_grad[0]      # not x.requires_grad: _chk may have returned a contiguous copy made under no_grad
        ctx.wshape = w.shape
        return y

    @staticmethod
    def backward(ctx, dy):
        x, w = ctx.saved_tensors
        dy = _chk(dy, "grad")
        K, N = x.shape[-1], dy.shape[-1]
        rows = x.numel() // K
        dw, db = _zeros_like_many([w, dy.new_empty(N)])
        dx = torch.empty_like(x) if ctx.need_dx else None
        with torch.cuda.device_of(x):
            _call("mmx_linear_bwd_prec", rows, K, N, _p(x), _p(w), _p(dy), _p(dw), _p(db), _p(dx), ctx.prec, _stream())
        return dx, dw.view(ctx.wshape), db, None


def linear(x, weight, bias, precision=None):
    """precision: None (follow ``set_precision``) | "fp32" | "tf32" (tensor cores, see mmx_linear_fwd_prec)."""
    return _Linear.apply(x, weight, bias, precision)


# ------------------------------------------------------------------------------------------------
# MixerBlock (mlp_mixer.py:138-164)
# ------------------------------------------------------------------------------------------------
_BLOCK_FIELDS = ("ln1_w", "ln1_b", "tok_w1", "tok_b1", "tok_w2", "tok_b2", "ln2_w", "ln2_b",
                 "ch_w1", "ch_b1", "ch_w2", "ch_b2", "se_w1", "se_w2")


def mlp_block_table(tensors):
    t = L.MmxMlpBlockParams()
    for f, v in zip(_BLOCK_FIELDS, tensors):
        setattr(t, f, _p(v))
    return t


_PRECISION = os.environ.get("MMX_PRECISION", "fp32")


def set_precision(precision):
    """Default arithmetic of the contractions inside the fused MixerBlock kernels: "fp32" (1e-5 parity with the
    reference) or "tf32" (tensor cores, 2e-3 parity).  A module's own ``precision`` attribute overrides it."""
    global _PRECISION
    if precision not in L.MMX_PREC:
        raise ValueError("unknown precision %r (expected one of %s)" % (precision, sorted(L.MMX_PREC)))
    _PRECISION = precision


def get_precision():
    return _PRECISION


# Device-resident dropout step counter for the autograd path (None: the host-side step of the modules is all there is).  A
# captured training step (rollout.RolloutTrainer) sets it and increments the tensor inside the graph, so every replay draws
# fresh masks although the host-side step value is frozen into the captured launches.
_STEP_DEV = None


def set_dropout_step_tensor(t):
    """t: int32 CUDA tensor with one element, or None."""
    global _STEP_DEV
    _STEP_DEV = t


def _step_dev_ptr(step_dev):
    if step_dev is not None:
        return step_dev
    return None if _STEP_DEV is None else _p(_STEP_DEV)


def mlp_block_desc(B, T, H, tok, ch, se_hidden, act, use_se, use_max, training, block_index, p, seed, step, precision=None,
                   step_dev=None):
    return L.MmxMlpBlockDesc(B, T, H, tok, ch, se_hidden, L.MMX_ACT[act], int(use_se), int(use_max), int(training),
                             block_index, L.MmxDropout(float(p), int(seed), int(step), _step_dev_ptr(step_dev)),
                             L.MMX_PREC[precision or _PRECISION])


class _MlpBlock(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, meta, *params):
        x = _chk(x, "x")
        params = [None if q is None else _chk(q, "parameter") for q in params]
        B, T, H = x.shape
        desc = mlp_block_desc(B, T, H, *meta)
        y = torch.empty_like(x)
        needs_grad = any(ctx.needs_input_grad)
        # the tcgen05 kernel family can hand the token-half output (+ SE gates) to the backward: one extra saved tile per
        # block instead of re-running the token half forward
        ctx.saved_x1 = bool(needs_grad and L.load().mmx_mlp_block_saves(C.byref(desc)))
        with torch.cuda.device_of(x):
            if ctx.saved_x1:
                x1 = torch.empty_like(x)
                gate = torch.empty(B, T, dtype=x.dtype, device=x.device)
                _call("mmx_mlp_block_fwd_save", C.byref(desc), C.byref(mlp_block_table(params)), _p(x), _p(y), _p(x1), _p(gate), _stream())
                ctx.save_for_backward(x, x1, gate, *[q for q in params if q is not None])
            else:
                _call("mmx_mlp_block_fwd", C.byref(desc), C.byref(mlp_block_table(params)), _p(x), _p(y), _stream())
                ctx.save_for_backward(x, *[q for q in params if q is not None])
        ctx.has = [q is not None for q in params]
        ctx.meta = meta
        return y

    @staticmethod
    def backward(ctx, dy):
        x, *rest = ctx.saved_tensors
        x1 = gate = None
        if ctx.saved_x1:
            x1, gate, *rest = rest
        it = iter(rest)
        params = [next(it) if h else None for h in ctx.has]
        dy = _chk(dy, "grad")
        B, T, H = x.shape
        desc = mlp_block_desc(B, T, H, *ctx.meta)
        grads = _zeros_like_many(params)
        dx = torch.empty_like(x)
        with torch.cuda.device_of(x):
            if ctx.saved_x1:
                _call("mmx_mlp_block_bwd_saved", C.byref(desc), C.byref(mlp_block_table(params)), C.byref(mlp_block_table(grads)),
                      _p(x), _p(x1), _p(gate), _p(dy), _p(dx), _stream())
            else:
                _call("mmx_mlp_block_bwd", C.byref(desc), C.byref(mlp_block_table(params)), C.byref(mlp_block_table(grads)),
                      _p(x), _p(dy), _p(dx), _stream())
        return (dx, None, *grads)


def mlp_block(x, meta, params):
    """meta = (tok, ch, se_hidden, act, use_se, use_max, training, block_index, p, seed, step, precision)."""
    return _MlpBlock.apply(x, meta, *params)


# ------------------------------------------------------------------------------------------------
# MixerBlock with BatchNorm1d inside the MLP blocks (regularization == -1, mlp_mixer.py:72-73, 88-94)
# ------------------------------------------------------------------------------------------------
class MlpBnBlock:
    """Static buffers + the stage-kernel sequence of one MixerBlock whose MlpBlocks regularise with BatchNorm1d.

    Batch statistics are global over the batch, so the block is a chain of stage kernels (include/mmx.h, csrc/mmx_api_bnmlp.cu)
    with a reduction between them; this class owns the saved tensors and is used both by the autograd Function below (fresh
    buffers per call) and by TrainStep (static buffers inside the captured graph).  Token MLP: BatchNorm1d(hidden_dim) on
    [B,H,*]; channel MLP: BatchNorm1d(seq_len) on [B,T,*]; reg1 after the activation, reg2 after fc2 (mlp_mixer.py:88-94).

    ``params`` = MixerBlock.kernel_params() (14, SE weights may be None); ``bns`` = the four BatchNorm1d modules in execution
    order (token reg1, token reg2, channel reg1, channel reg2).
    """

    def __init__(self, B, T, H, tok, ch, device, need_backward=True):
        e = lambda *shape: torch.empty(*shape, dtype=torch.float32, device=device)
        self.B, self.T, self.H, self.tok, self.ch = B, T, H, tok, ch
        self.nT, self.st1 = e(B, H, T), e(B * T, 2)
        self.u1, self.g1, self.v1 = e(B, H, tok), e(B, H, tok), e(B, H, T)
        self.x1 = e(B, T, H)
        self.n2, self.st2 = e(B, T, H), e(B * T, 2)
        self.u2, self.g2, self.v2 = e(B, T, ch), e(B, T, ch), e(B, T, H)
        self.bn = [torch.zeros(4 * c, dtype=torch.float32, device=device) for c in (H, H, T, T)]
        self.sums = torch.zeros(2 * max(H, T), dtype=torch.float64, device=device)
        self.trained = True
        if need_backward:
            self.coef = e(3 * max(H, T))
            self.dA, self.dC = e(B * T * H), e(B, T, H)
            self.dB = e(max(B * T * ch, B * H * tok))

    # channels / elements-per-channel of the four BatchNorm layers: (N, C, L, act?)
    def _geo(self, i):
        B, T, H, tok, ch = self.B, self.T, self.H, self.tok, self.ch
        return [(B, H, tok), (B, H, T), (B, T, ch), (B, T, H)][i]

    def _bn_vectors(self, i, u, act, bnm, training):
        """per-channel vectors of BatchNorm layer i for the tensor u (pre-activation when act >= 0)."""
        N, Cn, Ln = self._geo(i)
        st = _stream()
        if training:
            _call("mmx_bn1d_stats", N, Cn, Ln, act, _p(u), _p(self.sums), st)
            _call("mmx_bn_finalize", _p(self.sums), Cn, float(N * Ln), _p(bnm.weight), _p(bnm.bias), _p(bnm.running_mean), _p(bnm.running_var),
                  _p(bnm.num_batches_tracked), float(bnm.momentum if bnm.momentum is not None else 0.1), float(bnm.eps), _p(self.bn[i]), st)
        else:
            with torch.no_grad():
                xs = torch.rsqrt(bnm.running_var + bnm.eps)
                scale = bnm.weight.detach() * xs
                self.bn[i].copy_(torch.cat([scale, bnm.bias.detach() - bnm.running_mean * scale, xs, -bnm.running_mean * xs]))
        return self.bn[i]

    def forward(self, x, out, params, bns, act, se_hidden, use_max, training):
        (ln1w, ln1b, tw1, tb1, tw2, tb2, ln2w, ln2b, cw1, cb1, cw2, cb2, s1, s2) = params
        B, T, H, tok, ch = self.B, self.T, self.H, self.tok, self.ch
        st = _stream()
        a = L.MMX_ACT[act]
        self.trained = bool(training)
        # ---- token half: x1 = x + SE(BN(fc2(BN(act(fc1(LN1(x)^T)))))^T)
        _call("mmx_ln_fwd", B * T, H, T, _p(x), _p(ln1w), _p(ln1b), _p(self.nT), _p(self.st1), st)
        _call("mmx_linear_fwd", B * H, T, tok, _p(self.nT), _p(tw1), _p(tb1), _p(self.u1), st)
        bn = self._bn_vectors(0, self.u1, a, bns[0], training)
        _call("mmx_bn1d_apply", B, H, tok, a, _p(self.u1), _p(bn), _p(self.g1), st)
        _call("mmx_linear_fwd", B * H, tok, T, _p(self.g1), _p(tw2), _p(tb2), _p(self.v1), st)
        bn = self._bn_vectors(1, self.v1, -1, bns[1], training)
        _call("mmx_se_res_fwd", B, T, H, se_hidden, int(use_max), 1, 1, _p(x), _p(self.v1), _p(bn), _p(s1), _p(s2), _p(self.x1), st)
        # ---- channel half: out = x1 + SE(BN(fc2(BN(act(fc1(LN2(x1)))))))
        _call("mmx_ln_fwd", B * T, H, 0, _p(self.x1), _p(ln2w), _p(ln2b), _p(self.n2), _p(self.st2), st)
        _call("mmx_linear_fwd", B * T, H, ch, _p(self.n2), _p(cw1), _p(cb1), _p(self.u2), st)
        bn = self._bn_vectors(2, self.u2, a, bns[2], training)
        _call("mmx_bn1d_apply", B, T, ch, a, _p(self.u2), _p(bn), _p(self.g2), st)
        _call("mmx_linear_fwd", B * T, ch, H, _p(self.g2), _p(cw2), _p(cb2), _p(self.v2), st)
        bn = self._bn_vectors(3, self.v2, -1, bns[3], training)
        _call("mmx_se_res_fwd", B, T, H, se_hidden, int(use_max), 0, 0, _p(self.x1), _p(self.v2), _p(bn), _p(s1), _p(s2), _p(out), st)
        return out

    def _bn_backward(self, i, u, act, d, gw, gb):
        """d (gradient wrt the BatchNorm output, [N,C,L]) -> gradient wrt u, in place; gw / gb accumulated."""
        N, Cn, Ln = self._geo(i)
        st = _stream()
        _call("mmx_bn1d_bwd_reduce", N, Cn, Ln, act, _p(u), _p(self.bn[i]), _p(d), _p(self.sums), st)
        _call("mmx_bn_coef", _p(self.sums), Cn, float(N * Ln), _p(self.bn[i]), _p(self.coef), _p(gw), _p(gb), st)
        if not self.trained:               # eval mode: the statistics are constants, only the affine back-propagates
            self.coef[Cn:3 * Cn].zero_()
        _call("mmx_bn1d_bwd_apply", N, Cn, Ln, act, _p(u), _p(self.bn[i]), _p(self.coef), _p(d), _p(d), st)

    def backward(self, x, dout, dx, params, grads, bn_grads, act, se_hidden, use_max):
        """grads: tensors matching ``params`` (accumulated); bn_grads: [(d weight, d bias)] x 4 (accumulated)."""
        (ln1w, ln1b, tw1, tb1, tw2, tb2, ln2w, ln2b, cw1, cb1, cw2, cb2, s1, s2) = params
        (g_ln1w, g_ln1b, g_tw1, g_tb1, g_tw2, g_tb2, g_ln2w, g_ln2b, g_cw1, g_cb1, g_cw2, g_cb2, g_s1, g_s2) = grads
        B, T, H, tok, ch = self.B, self.T, self.H, self.tok, self.ch
        st = _stream()
        a = L.MMX_ACT[act]
        dA, dB, dC = self.dA, self.dB, self.dC
        # ---- channel half
        _call("mmx_se_res_bwd", B, T, H, se_hidden, int(use_max), 0, 0, _p(self.v2), _p(self.bn[3]), _p(s1), _p(s2), _p(dout),
              _p(g_s1), _p(g_s2), _p(dA), st)
        self._bn_backward(3, self.v2, -1, dA, *bn_grads[3])
        _call("mmx_linear_bwd", B * T, ch, H, _p(self.g2), _p(cw2), _p(dA), _p(g_cw2), _p(g_cb2), _p(dB), st)
        self._bn_backward(2, self.u2, a, dB, *bn_grads[2])
        _call("mmx_linear_bwd", B * T, H, ch, _p(self.n2), _p(cw1), _p(dB), _p(g_cw1), _p(g_cb1), _p(dA), st)
        _call("mmx_ln_bwd", B * T, H, 0, _p(self.x1), _p(self.st2), _p(ln2w), _p(dA), _p(dout), _p(dC), _p(g_ln2w), _p(g_ln2b), st)
        # ---- token half (dC = gradient wrt x1)
        _call("mmx_se_res_bwd", B, T, H, se_hidden, int(use_max), 1, 1, _p(self.v1), _p(self.bn[1]), _p(s1), _p(s2), _p(dC),
              _p(g_s1), _p(g_s2), _p(dA), st)
        self._bn_backward(1, self.v1, -1, dA, *bn_grads[1])
        _call("mmx_linear_bwd", B * H, tok, T, _p(self.g1), _p(tw2), _p(dA), _p(g_tw2), _p(g_tb2), _p(dB), st)
        self._bn_backward(0, self.u1, a, dB, *bn_grads[0])
        _call("mmx_linear_bwd", B * H, T, tok, _p(self.nT), _p(tw1), _p(dB), _p(g_tw1), _p(g_tb1), _p(dA), st)
        _call("mmx_ln_bwd", B * T, H, T, _p(x), _p(self.st1), _p(ln1w), _p(dA), _p(dC), _p(dx), _p(g_ln1w), _p(g_ln1b), st)
        return dx

    n_launches_fwd = 16      # training mode: 2 LN + 4 fc + 4 x (stats, finalize) + 2 apply + 2 SE
    n_launches_bwd = 22      # 2 SE + 4 x (reduce, coef, apply) + 4 fc + 2 LN


class _MlpBlockBN(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, meta, bns, *tensors):
        x = _chk(x, "x")
        params = [None if q is None else _chk(q, "parameter") for q in tensors[:14]]
        tok, ch, se_hidden, act, use_se, use_max, training = meta[:7]
        B, T, H = x.shape
        needs_grad = any(ctx.needs_input_grad)
        with torch.cuda.device_of(x):
            run = MlpBnBlock(B, T, H, tok, ch, x.device, need_backward=needs_grad)
            y = torch.empty_like(x)
            run.forward(x, y, params, bns, act, se_hidden if use_se else 0, use_max, training)
        ctx.run, ctx.params, ctx.x = run, params, x
        ctx.cfg = (act, se_hidden if use_se else 0, use_max)
        return y

    @staticmethod
    def backward(ctx, dy):
        dy = _chk(dy, "grad")
        run, params, x = ctx.run, ctx.params, ctx.x
        grads = _zeros_like_many(params)
        bn_flat = _zeros_like_many([run.bn[i][:run.bn[i].numel() // 4] for i in range(4) for _ in range(2)])
        bn_grads = [(bn_flat[2 * i], bn_flat[2 * i + 1]) for i in range(4)]
        dx = torch.empty_like(x)
        with torch.cuda.device_of(x):
            run.backward(x, dy, dx, params, grads, bn_grads, *ctx.cfg)
        ctx.run = None
        return (dx, None, None, *grads, *bn_flat)


def mlp_block_bn(x, meta, params, bns):
    """MixerBlock forward with BatchNorm1d regularisation.  ``bns``: the four BatchNorm1d modules (token reg1, token reg2,
    channel reg1, channel reg2); their weights / biases receive gradients, their running statistics are updated in training
    mode exactly as nn.BatchNorm1d does (momentum, unbiased variance, num_batches_tracked)."""
    bn_tensors = [t for m in bns for t in (m.weight, m.bias)]
    return _MlpBlockBN.apply(x, meta, tuple(bns), *params, *bn_tensors)


# ------------------------------------------------------------------------------------------------
# MlpMixer head (mlp_mixer.py:332-335)
# ------------------------------------------------------------------------------------------------
_HEAD_FIELDS = ("ln_w", "ln_b", "wt", "bt", "wf", "bf")


def mlp_head_table(tensors):
    t = L.MmxMlpHeadParams()
    for f, v in zip(_HEAD_FIELDS, tensors):
        setattr(t, f, _p(v))
    return t


class _MlpHead(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, ln_w, ln_b, wt, bt, wf, bf, precision):
        x = _chk(x, "x")
        ctx.prec = L.MMX_PREC[precision or _PRECISION]
        params = [_chk(q, "parameter") for q in (ln_w, ln_b, wt, bt, wf, bf)]
        B, T, H = x.shape
        To, D = bt.numel(), bf.numel()
        desc = L.MmxMlpHeadDesc(B, T, To, H, D)
        out = torch.empty(B, To, D, dtype=torch.float32, device=x.device)
        with torch.cuda.device_of(x):
            _call("mmx_mlp_head_fwd_prec", C.byref(desc), C.byref(mlp_head_table(params)), _p(x), _p(out), ctx.prec, _stream())
        ctx.save_for_backward(x, *params)
        return out

    @staticmethod
    def backward(ctx, dout):
        x, *params = ctx.saved_tensors
        dout = _chk(dout, "grad")
        B, T, H = x.shape
        To, D = params[3].numel(), params[5].numel()
        desc = L.MmxMlpHeadDesc(B, T, To, H, D)
        grads = _zeros_like_many(params)
        dx = torch.empty_like(x)
        with torch.cuda.device_of(x):
            _call("mmx_mlp_head_bwd_prec", C.byref(desc), C.byref(mlp_head_table(params)), C.byref(mlp_head_table(grads)),
                  _p(x), _p(dout), _p(dx), ctx.prec, _stream())
        return (dx, *grads, None)


def mlp_head(x, ln_w, ln_b, wt, bt, wf, bf, precision=None):
    return _MlpHead.apply(x, ln_w, ln_b, wt, bt, wf, bf, precision)


# ------------------------------------------------------------------------------------------------
# MPJPE (utils_mixer.py:48-53)
# ------------------------------------------------------------------------------------------------
class _Mpjpe(torch.autograd.Function):
    @staticmethod
    def forward(ctx, pred, gt):
        pred, gt = _chk(pred, "batch_pred"), _chk(gt, "batch_gt")
        if pred.numel() != gt.numel() or pred.numel() % 3:
            raise RuntimeError("mpjpe_error: shapes %s / %s are not matching [*, 3] joint arrays" % (tuple(pred.shape), tuple(gt.shape)))
        n = pred.numel() // 3
        loss_sum = torch.zeros(1, dtype=torch.float32, device=pred.device)
        dpred = torch.empty_like(pred) if ctx.needs_input_grad[0] else None
        with torch.cuda.device_of(pred):
            _call("mmx_mpjpe_fwd_bwd", _p(pred), _p(gt), _p(dpred), _p(loss_sum), n, 1.0, _stream())
        ctx.save_for_backward(dpred)
        return (loss_sum / n).reshape(())

    @staticmethod
    def backward(ctx, g):
        (dpred,) = ctx.saved_tensors
        return dpred * g, None


def mpjpe_error(batch_pred, batch_gt):
    """Drop-in for ``h36m.utils.utils_mixer.mpjpe_error`` (one fused kernel: loss + dL/dpred)."""
    return _Mpjpe.apply(batch_pred, batch_gt)


class _AngleL1(torch.autograd.Function):
    @staticmethod
    def forward(ctx, pred, gt):
        pred, gt = _chk(pred, "prediction"), _chk(gt, "target")
        if pred.numel() != gt.numel() or gt.dim() < 1:
            raise RuntimeError("angle_l1_error: shapes %s / %s do not match" % (tuple(pred.shape), tuple(gt.shape)))
        D = gt.shape[-1]
        rows = gt.numel() // D
        loss_sum = torch.zeros(1, dtype=torch.float32, device=pred.device)
        dpred = torch.empty_like(pred) if ctx.needs_input_grad[0] else None
        with torch.cuda.device_of(pred):
            _call("mmx_l1_fwd_bwd", _p(pred), _p(gt), _p(dpred), _p(loss_sum), rows, D, 1.0, _stream())
        ctx.save_for_backward(dpred)
        return (loss_sum / rows).reshape(())

    @staticmethod
    def backward(ctx, g):
        (dpred,) = ctx.saved_tensors
        return dpred * g, None


def angle_l1_error(pred, gt):
    """The reference's joint-angle training loss, ``torch.mean(torch.sum(torch.abs(pred.reshape(-1, out_n, D) - gt), dim=2).view(-1))``
    (train_mixer_h36m.py:187, train_autoreg_mixer_h36m.py:209-210), as one fused kernel (loss + dL/dpred).  ``gt``: [..., D]."""
    return _AngleL1.apply(pred, gt)


# ------------------------------------------------------------------------------------------------
# ConvMixer (conv_mixer_model.py, positional_encoder.py)
# ------------------------------------------------------------------------------------------------
def conv_half_table(tensors, bn_aff=None):
    """tensors: (ln_w, ln_b, conv_w, conv_b, se_w1, se_w2) — the order of ``MmxConvHalfParams``; ``bn_aff``: optional
    eval-mode BatchNorm affine [scale | shift] (2C floats)."""
    t = L.MmxConvHalfParams()
    for f, v in zip(("ln_w", "ln_b", "conv_w", "conv_b", "se_w1", "se_w2"), tensors):
        setattr(t, f, _p(v))
    t.bn_aff = _p(bn_aff)
    return t


def conv_half_desc(B, C, T, E, kernel, pad, se_hidden, act, use_se, use_max, training, site, p, seed, step, step_dev=None):
    return L.MmxConvHalfDesc(B, C, T, E, kernel[0], kernel[1], pad[0], pad[1], se_hidden, L.MMX_ACT[act], int(use_se),
                             int(use_max), int(training), site, L.MmxDropout(float(p), int(seed), int(step), _step_dev_ptr(step_dev)))


class _ConvHalf(torch.autograd.Function):
    """One half of ConvMixerBlock.forward (conv_mixer_model.py:279-284 / :287-292): y = x + SE(reg(act(conv(LN(x)))))."""

    @staticmethod
    def forward(ctx, x, meta, *params):
        x = _chk(x, "x")
        params = [None if q is None else _chk(q, "parameter") for q in params]
        B, C, T, E = x.shape
        desc = conv_half_desc(B, C, T, E, *meta)
        y = torch.empty_like(x)
        with torch.cuda.device_of(x):
            _call("mmx_conv_half_fwd", C_.byref(desc), C_.byref(conv_half_table(params)), _p(x), _p(y), _stream())
        ctx.save_for_backward(x, *[q for q in params if q is not None])
        ctx.has = [q is not None for q in params]
        ctx.meta = meta
        return y

    @staticmethod
    def backward(ctx, dy):
        x, *rest = ctx.saved_tensors
        it = iter(rest)
        params = [next(it) if h else None for h in ctx.has]
        dy = _chk(dy, "grad")
        B, C, T, E = x.shape
        desc = conv_half_desc(B, C, T, E, *ctx.meta)
        grads = _zeros_like_many(params)
        dx = torch.empty_like(x)
        with torch.cuda.device_of(x):
            _call("mmx_conv_half_bwd", C_.byref(desc), C_.byref(conv_half_table(params)), C_.byref(conv_half_table(grads)),
                  _p(x), _p(dy), _p(dx), _stream())
        return (dx, None, *grads)


def conv_half(x, meta, params, bn_aff=None):
    """meta = (kernel, pad, se_hidden, act, use_se, use_max, training, site, p, seed, step).  ``bn_aff``: eval-mode
    BatchNorm folded to [scale | shift] (treated as a constant: no gradient flows to the BN parameters in eval mode)."""
    if bn_aff is None:
        return _ConvHalf.apply(x, meta, *params)
    return _ConvHalfAffine.apply(x, meta, bn_aff, *params)


class _ConvHalfAffine(torch.autograd.Function):
    """The fused half with a constant per-channel affine after the activation (BatchNorm2d in eval mode)."""

    @staticmethod
    def forward(ctx, x, meta, aff, *params):
        x, aff = _chk(x, "x"), _chk(aff, "bn affine")
        params = [None if q is None else _chk(q, "parameter") for q in params]
        B, C, T, E = x.shape
        desc = conv_half_desc(B, C, T, E, *meta)
        y = torch.empty_like(x)
        with torch.cuda.device_of(x):
            _call("mmx_conv_half_fwd", C_.byref(desc), C_.byref(conv_half_table(params, aff)), _p(x), _p(y), _stream())
        ctx.save_for_backward(x, aff, *[q for q in params if q is not None])
        ctx.has = [q is not None for q in params]
        ctx.meta = meta
        return y

    @staticmethod
    def backward(ctx, dy):
        x, aff, *rest = ctx.saved_tensors
        it = iter(rest)
        params = [next(it) if h else None for h in ctx.has]
        dy = _chk(dy, "grad")
        B, C, T, E = x.shape
        desc = conv_half_desc(B, C, T, E, *ctx.meta)
        grads = _zeros_like_many(params)
        dx = torch.empty_like(x)
        with torch.cuda.device_of(x):
            _call("mmx_conv_half_bwd", C_.byref(desc), C_.byref(conv_half_table(params, aff)), C_.byref(conv_half_table(grads)),
                  _p(x), _p(dy), _p(dx), _stream())
        return (dx, None, None, *grads)


# ---- training-mode BatchNorm2d between the activation and the SE layer (regularization == -1) ----------------
BN_EPS = 1e-5


def bn_forward_passes(desc, tw, x, z, y, sums, bn, bn_w, bn_b, running_mean, running_var, num_batches_tracked, momentum=0.1):
    """statistics pass -> mmx_bn_finalize (per-channel vectors, running statistics as nn.BatchNorm2d: biased variance to
    normalise, unbiased for the running estimate) -> apply pass.  ``sums`` (float64 [2C]) must be zero on entry and is zero
    again on exit; ``bn`` (float32 [4C]) receives [scale | shift | xs | xo]."""
    B, Cn, T, E = x.shape
    st = _stream()
    _call("mmx_conv_half_bn_stats", C_.byref(desc), C_.byref(tw), _p(x), _p(z), _p(sums), st)
    _call("mmx_bn_finalize", _p(sums), Cn, float(B * T * E), _p(bn_w), _p(bn_b), _p(running_mean), _p(running_var),
          _p(num_batches_tracked), float(momentum), BN_EPS, _p(bn), st)
    _call("mmx_conv_half_bn_apply", C_.byref(desc), C_.byref(tw), _p(bn), _p(x), _p(z), _p(y), st)
    return bn


def bn_backward_passes(desc, tw, tg, x, z, dy, dx, bn, gd, sums, coef, gw, gb, n):
    """pass 1 (SE backward + batch sums) -> mmx_bn_coef (coefficients; gw += d bn.weight, gb += d bn.bias) -> pass 2 (BN / conv /
    LN backward).  ``sums`` zero on entry and on exit."""
    Cn = bn.numel() // 4
    st = _stream()
    _call("mmx_conv_half_bn_bwd1", C_.byref(desc), C_.byref(tw), C_.byref(tg), _p(bn), _p(z), _p(dy), _p(gd), _p(sums), st)
    _call("mmx_bn_coef", _p(sums), Cn, float(n), _p(bn), _p(coef), _p(gw), _p(gb), st)
    _call("mmx_conv_half_bn_bwd2", C_.byref(desc), C_.byref(tw), C_.byref(tg), _p(bn), _p(coef), _p(x), _p(z), _p(dy), _p(gd), _p(dx), st)


class _ConvHalfBN(torch.autograd.Function):
    """One half with training-mode BatchNorm2d: y = x + SE(BN(act(conv(LN(x)))))  (conv_mixer_model.py:139-141,279-292)."""

    @staticmethod
    def forward(ctx, x, meta, bn_w, bn_b, running_mean, running_var, num_batches_tracked, *params):
        x = _chk(x, "x")
        params = [None if q is None else _chk(q, "parameter") for q in params]
        bn_w, bn_b = _chk(bn_w, "bn weight"), _chk(bn_b, "bn bias")
        B, C, T, E = x.shape
        desc = conv_half_desc(B, C, T, E, *meta)
        z, y = torch.empty_like(x), torch.empty_like(x)
        sums = torch.zeros(2 * C, dtype=torch.float64, device=x.device)
        bn = torch.empty(4 * C, dtype=torch.float32, device=x.device)
        with torch.cuda.device_of(x):
            bn_forward_passes(desc, conv_half_table(params), x, z, y, sums, bn, bn_w, bn_b, running_mean, running_var, num_batches_tracked)
        ctx.save_for_backward(x, z, bn, *[q for q in params if q is not None])
        ctx.has = [q is not None for q in params]
        ctx.meta = meta
        return y

    @staticmethod
    def backward(ctx, dy):
        x, z, bn, *rest = ctx.saved_tensors
        it = iter(rest)
        params = [next(it) if h else None for h in ctx.has]
        dy = _chk(dy, "grad")
        B, C, T, E = x.shape
        desc = conv_half_desc(B, C, T, E, *ctx.meta)
        grads = _zeros_like_many(params)
        dx = torch.empty_like(x)
        gd = torch.empty(B, T, 2, dtype=torch.float32, device=x.device)
        sums = torch.zeros(2 * C, dtype=torch.float64, device=x.device)
        coef = torch.empty(3 * C, dtype=torch.float32, device=x.device)
        dw, db = torch.zeros(C, dtype=torch.float32, device=x.device), torch.zeros(C, dtype=torch.float32, device=x.device)
        with torch.cuda.device_of(x):
            bn_backward_passes(desc, conv_half_table(params), conv_half_table(grads), x, z, dy, dx, bn, gd, sums, coef, dw, db, B * T * E)
        return (dx, None, dw, db, None, None, None, *grads)


def conv_half_bn(x, meta, bn_module, params):
    return _ConvHalfBN.apply(x, meta, bn_module.weight, bn_module.bias, bn_module.running_mean, bn_module.running_var,
                             bn_module.num_batches_tracked, *params)


def bn_eval_affine(bn_module):
    """BatchNorm2d in eval mode as [scale | shift] (2C floats)."""
    scale = bn_module.weight.detach() * torch.rsqrt(bn_module.running_var + bn_module.eps)
    return torch.cat([scale, bn_module.bias.detach() - bn_module.running_mean * scale]).contiguous()


# ---- large halves: shapes the fused kernels do not serve (mmx_conv_half_plan), BatchNorm with the max squeeze ----------------
def conv_prec(precision):
    """MMX_PREC_* of a ConvMixer convolution.  ``None`` is fp32: unlike the MlpMixer, the ConvMixer does not follow
    ``set_precision`` / MMX_PRECISION (ConvMixer runs under those settings have always been fp32 and stay bit for bit); it opts
    in through ``ConvMixer.set_precision("tf32")``."""
    return L.MMX_PREC[precision or "fp32"]


def conv_tc5_serves(B, C, T, E, meta):
    """True when precision "tf32" runs this half's convolutions on tcgen05 (mmx_conv2d_tc5_serves)."""
    return bool(L.load().mmx_conv2d_tc5_serves(C_.byref(conv_half_desc(B, C, T, E, *meta))))


def conv_half_fits(B, C, T, E, meta):
    """True when the fused half kernels (forward and backward) serve this shape; else the stage-kernel chain below runs."""
    desc = conv_half_desc(B, C, T, E, *meta)
    lib = L.load()
    return lib.mmx_conv_half_plan(C_.byref(desc), 0, None, None) == 0 and lib.mmx_conv_half_plan(C_.byref(desc), 1, None, None) == 0


class ConvHalfLarge:
    """Static buffers + the stage-kernel sequence of one ConvMixerBlock half that does not fit the fused kernels (include/mmx.h,
    csrc/mmx_api_conv_large.cu): LN -> conv2d -> [BatchNorm statistics] -> act / reg / SE / residual, intermediates in HBM.
    Used by the autograd Function below (fresh buffers per call) and by TrainStep (static buffers inside the captured graph).
    ``params`` = ConvMixerBlock.half_params(half); ``bn``: the half's BatchNorm2d module or None."""

    def __init__(self, B, C, T, E, device, need_backward=True, with_bn=False, precision=None):
        e = lambda *shape: torch.empty(*shape, dtype=torch.float32, device=device)
        self.B, self.C, self.T, self.E = B, C, T, E
        self.prec = conv_prec(precision)
        self.n, self.stats, self.z = e(B, C, T, E), e(B * C * T, 2), e(B, C, T, E)
        self.bn = torch.zeros(4 * C, dtype=torch.float32, device=device) if with_bn else None
        self.sums = torch.zeros(2 * C, dtype=torch.float64, device=device) if with_bn else None
        self.trained = True
        if need_backward:
            self.gd, self.dz, self.dn = e(B, T, 3), e(B, C, T, E), e(B, C, T, E)
            self.coef = e(3 * C) if with_bn else None

    def forward(self, desc, x, y, params, bnm=None):
        ln_w, ln_b, cw, cb, s1, s2 = params
        B, Cn, T, E = self.B, self.C, self.T, self.E
        st = _stream()
        _call("mmx_ln_fwd", B * Cn * T, E, 0, _p(x), _p(ln_w), _p(ln_b), _p(self.n), _p(self.stats), st)
        _call("mmx_conv2d_large_fwd_prec", C_.byref(desc), 0, _p(self.n), _p(cw), _p(cb), _p(self.z), self.prec, st)
        aff = None
        self.trained = bool(desc.training)
        if bnm is not None:
            if desc.training:
                _call("mmx_bn1d_stats", B, Cn, T * E, desc.act, _p(self.z), _p(self.sums), st)
                _call("mmx_bn_finalize", _p(self.sums), Cn, float(B * T * E), _p(bnm.weight), _p(bnm.bias), _p(bnm.running_mean),
                      _p(bnm.running_var), _p(bnm.num_batches_tracked), float(bnm.momentum if bnm.momentum is not None else 0.1),
                      float(bnm.eps), _p(self.bn), st)
            else:
                with torch.no_grad():
                    xs = torch.rsqrt(bnm.running_var + bnm.eps)
                    scale = bnm.weight.detach() * xs
                    self.bn.copy_(torch.cat([scale, bnm.bias.detach() - bnm.running_mean * scale, xs, -bnm.running_mean * xs]))
            aff = self.bn
        _call("mmx_conv_tail_fwd", C_.byref(desc), _p(x), _p(self.z), _p(aff), _p(s1), _p(s2), _p(y), st)
        return y

    def backward(self, desc, x, dy, dx, params, grads, bn_grads=None):
        ln_w, ln_b, cw, cb, s1, s2 = params
        g_ln_w, g_ln_b, g_cw, g_cb, g_s1, g_s2 = grads
        B, Cn, T, E = self.B, self.C, self.T, self.E
        st = _stream()
        bn = self.bn if bn_grads is not None else None
        _call("mmx_conv_tail_bwd1", C_.byref(desc), _p(self.z), _p(dy), _p(bn), _p(s1), _p(s2), _p(g_s1), _p(g_s2), _p(self.gd),
              _p(self.sums) if bn is not None else None, st)
        coef = None
        if bn is not None:
            _call("mmx_bn_coef", _p(self.sums), Cn, float(B * T * E), _p(self.bn), _p(self.coef), _p(bn_grads[0]), _p(bn_grads[1]), st)
            if not self.trained:
                self.coef[Cn:3 * Cn].zero_()
            coef = self.coef
        _call("mmx_conv_tail_bwd2", C_.byref(desc), _p(self.z), _p(dy), _p(self.gd), _p(bn), _p(coef), _p(self.dz), st)
        _call("mmx_conv2d_large_wgrad_prec", C_.byref(desc), _p(self.dz), _p(self.n), _p(g_cw), _p(g_cb), self.prec, st)
        _call("mmx_conv2d_large_fwd_prec", C_.byref(desc), 1, _p(self.dz), _p(cw), None, _p(self.dn), self.prec, st)
        _call("mmx_ln_bwd", B * Cn * T, E, 0, _p(x), _p(self.stats), _p(ln_w), _p(self.dn), _p(dy), _p(dx), _p(g_ln_w), _p(g_ln_b), st)
        return dx

    @staticmethod
    def launches(with_bn):
        return (5 if with_bn else 3), (7 if with_bn else 6)


class _ConvHalfLarge(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, meta, bnm, precision, *tensors):
        x = _chk(x, "x")
        params = [None if q is None else _chk(q, "parameter") for q in tensors[:6]]
        B, C, T, E = x.shape
        desc = conv_half_desc(B, C, T, E, *meta)
        needs_grad = any(ctx.needs_input_grad)
        with torch.cuda.device_of(x):
            run = ConvHalfLarge(B, C, T, E, x.device, need_backward=needs_grad, with_bn=bnm is not None, precision=precision)
            y = torch.empty_like(x)
            run.forward(desc, x, y, params, bnm)
        ctx.run, ctx.params, ctx.x, ctx.meta, ctx.has_bn = run, params, x, meta, bnm is not None
        return y

    @staticmethod
    def backward(ctx, dy):
        dy = _chk(dy, "grad")
        run, params, x = ctx.run, ctx.params, ctx.x
        B, C, T, E = x.shape
        desc = conv_half_desc(B, C, T, E, *ctx.meta)
        grads = _zeros_like_many(params)
        bn_grads = None
        if ctx.has_bn:
            bn_grads = [torch.zeros(C, dtype=torch.float32, device=x.device), torch.zeros(C, dtype=torch.float32, device=x.device)]
        dx = torch.empty_like(x)
        with torch.cuda.device_of(x):
            run.backward(desc, x, dy, dx, params, grads, bn_grads)
        ctx.run = None
        return (dx, None, None, None, *grads, *(bn_grads or []))


def conv_half_large(x, meta, params, bn_module=None, precision=None):
    """One ConvMixerBlock half through the stage-kernel chain (large shapes; BatchNorm with max squeeze).  ``precision``: see
    ``conv_prec``."""
    extra = [bn_module.weight, bn_module.bias] if bn_module is not None else []
    return _ConvHalfLarge.apply(x, meta, bn_module, precision, *params, *extra)


class _SeTail(torch.autograd.Function):
    """mode_conv='once': y = x + se(x), or 2x without SE (conv_mixer_model.py:259-263,287-292)."""

    @staticmethod
    def forward(ctx, x, meta, se_w1, se_w2):
        x = _chk(x, "x")
        se_hidden, use_se, use_max = meta
        if use_se:
            se_w1, se_w2 = _chk(se_w1, "se weight"), _chk(se_w2, "se weight")
        B, C, T, E = x.shape
        y = torch.empty_like(x)
        with torch.cuda.device_of(x):
            _call("mmx_se_tail_fwd", B, C, T, E, se_hidden, int(use_se), int(use_max), _p(se_w1), _p(se_w2), _p(x), _p(y), _stream())
        if use_se:
            ctx.save_for_backward(x, se_w1, se_w2)
        else:
            ctx.save_for_backward(x)
        ctx.meta = meta
        return y

    @staticmethod
    def backward(ctx, dy):
        se_hidden, use_se, use_max = ctx.meta
        x, *se = ctx.saved_tensors
        dy = _chk(dy, "grad")
        B, C, T, E = x.shape
        g1 = g2 = None
        if use_se:
            g1, g2 = _zeros_like_many(se)
        dx = torch.empty_like(x)
        with torch.cuda.device_of(x):
            _call("mmx_se_tail_bwd", B, C, T, E, se_hidden, int(use_se), int(use_max), _p(se[0]) if use_se else None,
                  _p(se[1]) if use_se else None, _p(g1), _p(g2), _p(x), _p(dy), _p(dx), _stream())
        return dx, None, g1, g2


def se_tail(x, se_hidden, use_se, use_max, se_w1, se_w2):
    return _SeTail.apply(x, (se_hidden, use_se, use_max), se_w1, se_w2)


def encoder_table(tensors):
    t = L.MmxEncoderParams()
    for f, v in zip(("freq", "w", "b", "wc", "bc"), tensors):
        setattr(t, f, _p(v))
    return t


class _PoseEncoder(torch.autograd.Function):
    """PoseEncoder.forward (positional_encoder.py:79-97)."""

    @staticmethod
    def forward(ctx, x, n_harmonic, C, freq, w, b, wc, bc):
        x, w, b, wc, bc = _chk(x, "x"), _chk(w, "weight"), _chk(b, "bias"), _chk(wc, "weight"), _chk(bc, "bias")
        if n_harmonic > 0:
            freq = _chk(freq, "frequencies")
        B, T, D = x.shape
        E = b.numel()
        desc = L.MmxEncoderDesc(B, T, D, E, C, n_harmonic)
        m = torch.empty(B * T, E, dtype=torch.float32, device=x.device)
        y = torch.empty(B, C, T, E, dtype=torch.float32, device=x.device)
        with torch.cuda.device_of(x):
            _call("mmx_pose_encoder_fwd", C_.byref(desc), C_.byref(encoder_table([freq, w, b, wc, bc])), _p(x), _p(m), _p(y), _stream())
        ctx.save_for_backward(x, m, w, b, wc, bc, *([freq] if n_harmonic > 0 else []))
        ctx.dims = (B, T, D, E, C, n_harmonic)
        ctx.need_dx = ctx.needs_input_grad[0]
        return y

    @staticmethod
    def backward(ctx, dy):
        x, m, w, b, wc, bc, *fr = ctx.saved_tensors
        freq = fr[0] if fr else None
        dy = _chk(dy, "grad")
        B, T, D, E, C, Hn = ctx.dims
        desc = L.MmxEncoderDesc(B, T, D, E, C, Hn)
        gw, gb, gwc, gbc = _zeros_like_many([w, b, wc, bc])
        dm = torch.empty_like(m)
        dx = torch.empty_like(x) if ctx.need_dx else None
        with torch.cuda.device_of(x):
            _call("mmx_pose_encoder_bwd", C_.byref(desc), C_.byref(encoder_table([freq, w, b, wc, bc])),
                  C_.byref(encoder_table([None, gw, gb, gwc, gbc])), _p(x), _p(m), _p(dy), _p(dm), _p(dx), _stream())
        return dx, None, None, None, gw, gb, gwc, gbc


def pose_encoder(x, n_harmonic, C, freq, w, b, wc, bc):
    return _PoseEncoder.apply(x, n_harmonic, C, freq, w, b, wc, bc)


def conv_head_table(tensors):
    t = L.MmxConvHeadParams()
    for f, v in zip(("ln_w", "ln_b", "wt", "bt", "wp", "bp", "wf", "bf"), tensors):
        setattr(t, f, _p(v))
    return t


class _ConvHead(torch.autograd.Function):
    """LN -> conv_out -> project_channels -> GELU -> fc_out (conv_mixer_model.py:455-463)."""

    @staticmethod
    def forward(ctx, y, *params):
        y = _chk(y, "y")
        params = [_chk(q, "parameter") for q in params]
        B, C, T, E = y.shape
        To, D = params[3].numel(), params[7].numel()
        desc = L.MmxConvHeadDesc(B, C, T, To, E, D)
        out = torch.empty(B, To, D, dtype=torch.float32, device=y.device)
        with torch.cuda.device_of(y):
            _call("mmx_conv_head_fwd", C_.byref(desc), C_.byref(conv_head_table(params)), _p(y), _p(out), _stream())
        ctx.save_for_backward(y, *params)
        return out

    @staticmethod
    def backward(ctx, dout):
        y, *params = ctx.saved_tensors
        dout = _chk(dout, "grad")
        B, C, T, E = y.shape
        To, D = params[3].numel(), params[7].numel()
        desc = L.MmxConvHeadDesc(B, C, T, To, E, D)
        grads = _zeros_like_many(params)
        dy = torch.empty_like(y)
        with torch.cuda.device_of(y):
            _call("mmx_conv_head_bwd", C_.byref(desc), C_.byref(conv_head_table(params)), C_.byref(conv_head_table(grads)),
                  _p(y), _p(dout), _p(dy), _stream())
        return (dy, *grads)


def conv_head(y, ln_w, ln_b, wt, bt, wp, bp, wf, bf):
    return _ConvHead.apply(y, ln_w, ln_b, wt, bt, wp, bp, wf, bf)


# ------------------------------------------------------------------------------------------------
# the callers either side of model(x): step input (train_mixer_h36m.py:117-120,179), PCK / AUC (utils_mixer.py:20-45)
# ------------------------------------------------------------------------------------------------
def window_split(batch, dim_used, input_n, output_n, x_scale=1.0, gt_scale=1.0, out=None):
    """``(batch[:, :input_n, dim_used] * x_scale, batch[:, input_n:input_n+output_n, dim_used] * gt_scale)`` in one pass over
    the raw window.  ``dim_used``: int32 CUDA tensor (or anything convertible).  ``out``: optional preallocated (x, gt)."""
    batch = _chk(batch, "batch")
    if not isinstance(dim_used, torch.Tensor):
        dim_used = torch.as_tensor(dim_used, dtype=torch.int32)
    dim_used = dim_used.to(device=batch.device, dtype=torch.int32).contiguous()
    B, Ttot, Dfull = batch.shape
    D = dim_used.numel()
    x, gt = out if out is not None else (torch.empty(B, input_n, D, device=batch.device), torch.empty(B, output_n, D, device=batch.device))
    with torch.cuda.device_of(batch):
        _call("mmx_window_split", _p(batch), B, Ttot, Dfull, _p(dim_used), D, input_n, output_n, float(x_scale), float(gt_scale),
              _p(x), _p(gt), _stream())
    return x, gt


_PCK_THRESH = {}


def auc_pck_metric(predictions, targets):
    """Drop-in for ``h36m.utils.utils_mixer.auc_pck_metric``: area under the PCK curve for thresholds 0.001 ... 0.299.
    One kernel builds the distance histogram over the 299 thresholds (the reference runs 299 x 6 elementwise kernels); the
    cumulative sum and the trapezoid rule are tensor ops on 300 elements.  No host synchronisation."""
    import numpy as np
    pred, gt = _chk(predictions, "predictions"), _chk(targets, "targets")
    if pred.shape != gt.shape or pred.shape[-1] != 3:
        raise RuntimeError("auc_pck_metric: expected two tensors of the same shape (..., n_joints, 3)")
    dev = pred.device
    th = _PCK_THRESH.get(dev)
    if th is None:
        th = _PCK_THRESH[dev] = torch.from_numpy(np.arange(0.001, 0.3, 0.001).astype(np.float32)).to(dev)
    n = th.numel()
    nj = pred.numel() // 3
    hist = torch.zeros(n + 1, dtype=torch.int32, device=dev)
    with torch.cuda.device_of(pred):
        _call("mmx_pck_hist", _p(pred), _p(gt), nj, _p(th), n, _p(hist), _stream())
    pck_values = torch.cumsum(hist[:n], 0).to(torch.float32) / float(nj)
    return torch.trapz(pck_values, dx=0.001) / 0.299
