"""Host-side runners over the libmmx C ABI (include/mmx.h), and the autograd Function that applies them.

A runner is one layer's kernel sequence: the embedding, a MixerBlock, a ConvMixerBlock half, the SE tail, an encoder or a
head.  It is built once from the module, the batch size, the device and whether a backward follows; it makes its routing
decision (which kernels, which saved intermediates) in its constructor and owns those intermediates.  ``forward(x, y,
training)`` and ``backward(x, dy, dx, grads)`` launch its kernels; ``launches`` counts them (forward, backward).  The same
runners serve both host paths: ``model(x)`` builds fresh ones per call and applies each through ``_Layer`` (autograd), and
``train.TrainStep`` builds them once per batch size over static buffers and the flat gradient bucket.

Every op launches hand-written sm_100a kernels on ``torch.cuda.current_stream()``; inputs must be CUDA fp32 tensors.  There
is no CPU / eager-PyTorch implementation: non-CUDA input raises.  Backward runs on PyTorch's autograd worker thread — the C
ABI holds no thread-local CUDA state and takes the stream explicitly, and we re-enter the tensor's device before every call.
"""
from __future__ import annotations

import ctypes as C
import os

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
    ref = next((t for t in tensors if t is not None), None)
    if ref is None:
        return list(tensors)
    flat = torch.zeros(sum(sizes), dtype=torch.float32, device=ref.device)
    out, o = [], 0
    for t, n in zip(tensors, sizes):
        out.append(None if t is None else flat[o:o + t.numel()].view(t.shape))
        o += n
    return out


def _call(name, *args):
    lib = L.load()
    L.check(lib, getattr(lib, name)(*args), name)


def _empty(device):
    return lambda *shape: torch.empty(*shape, dtype=torch.float32, device=device)


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
# precision, dropout, and one layer through autograd
# ------------------------------------------------------------------------------------------------
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


def dropout_source(block):
    """(seed, step, step_dev) of one autograd call of a Mixer / ConvMixer block: the masks follow ``torch.initial_seed()`` and
    the block's call count, which advances once per training call with dropout; step_dev None reads ``set_dropout_step_tensor``."""
    if not (block.training and block.regularization > 0.0):
        return 0, 0, None
    step = block._calls
    block._calls = (block._calls + 1) & 0xFFFFFFFF
    return torch.initial_seed() & 0xFFFFFFFFFFFFFFFF, step, None


class _Layer(torch.autograd.Function):
    """One runner as one autograd node.  The input and the parameters are saved through ``save_for_backward`` (so autograd's
    in-place-modification check covers them); the runner holds its own intermediates until the backward."""

    @staticmethod
    def forward(ctx, run, training, x, *params):
        x = _chk(x, "x")
        for q in params:
            if q is not None:
                _chk(q, "parameter")
        y = torch.empty(run.out_shape, dtype=torch.float32, device=x.device)
        with torch.cuda.device_of(x):
            run.forward(x, y, training)
        ctx.run = run
        ctx.save_for_backward(x, *params)
        return y

    @staticmethod
    def backward(ctx, dy):
        x, *params = ctx.saved_tensors
        dy = _chk(dy, "grad")
        grads = _zeros_like_many(params)
        dx = torch.empty_like(x) if ctx.needs_input_grad[2] or not ctx.run.optional_dx else None
        with torch.cuda.device_of(x):
            ctx.run.backward(x, dy, dx, grads)
        ctx.run = None
        return (None, None, dx, *grads)


def forward_layers(module, x):
    """``module(x)`` through autograd: the module's runners, built fresh for this call, one autograd node each."""
    need_backward = torch.is_grad_enabled() and (x.requires_grad or any(p.requires_grad for p in module.parameters()))
    for run in module.runners(x.shape[0], x.device, need_backward):
        x = _Layer.apply(run, module.training, x, *run.params)
    return x


class _Runner:
    optional_dx = False     # True: the first layer, whose input gradient is computed only when asked for
    launches = (1, 1)


def bn_vectors(bnm, training, sums, count, out):
    """Per-channel vectors [scale | shift | xs | xo] (4C floats) of the BatchNorm module ``bnm`` into ``out``.  Training: from
    the batch sums ``sums`` (float64 [2C], zero on entry and again on exit) over ``count`` elements per channel, by
    mmx_bn_finalize, which also updates the running statistics as nn.BatchNorm does (biased variance to normalise, unbiased
    for the running estimate, momentum, num_batches_tracked).  Eval: from the running statistics; the first 2C floats are then
    the constant affine [scale | shift] that the fused ConvMixer kernels apply."""
    if training:
        _call("mmx_bn_finalize", _p(sums), out.numel() // 4, float(count), _p(bnm.weight), _p(bnm.bias), _p(bnm.running_mean),
              _p(bnm.running_var), _p(bnm.num_batches_tracked), float(bnm.momentum if bnm.momentum is not None else 0.1),
              float(bnm.eps), _p(out), _stream())
    else:
        with torch.no_grad():
            xs = torch.rsqrt(bnm.running_var + bnm.eps)
            scale = bnm.weight.detach() * xs
            out.copy_(torch.cat([scale, bnm.bias.detach() - bnm.running_mean * scale, xs, -bnm.running_mean * xs]))
    return out


# ------------------------------------------------------------------------------------------------
# MlpMixer: embedding, MixerBlock (mlp_mixer.py:138-164), head
# ------------------------------------------------------------------------------------------------
class LinearEmbed(_Runner):
    """MlpMixer.conv: Conv2d(1, H, (1, D)) is a per-frame Linear D -> H (mlp_mixer.py:325-327)."""
    optional_dx = True

    def __init__(self, model, B, device, need_backward):
        self.model = model
        self.params = [model.conv.weight, model.conv.bias]
        self.dims = (B * model.seq_len, model.input_size, model.hidden_dim)
        self.in_shape, self.out_shape = (B, model.seq_len, model.input_size), (B, model.seq_len, model.hidden_dim)

    def forward(self, x, y, training):
        w, b = self.params
        self.prec = L.MMX_PREC[self.model.precision or _PRECISION]
        _call("mmx_linear_fwd_prec", *self.dims, _p(x), _p(w), _p(b), _p(y), self.prec, _stream())

    def backward(self, x, dy, dx, grads):
        _call("mmx_linear_bwd_prec", *self.dims, _p(x), _p(self.params[0]), _p(dy), _p(grads[0]), _p(grads[1]), _p(dx), self.prec, _stream())


_BLOCK_FIELDS = ("ln1_w", "ln1_b", "tok_w1", "tok_b1", "tok_w2", "tok_b2", "ln2_w", "ln2_b",
                 "ch_w1", "ch_b1", "ch_w2", "ch_b2", "se_w1", "se_w2")


def mlp_block_table(tensors):
    t = L.MmxMlpBlockParams()
    for f, v in zip(_BLOCK_FIELDS, tensors):
        setattr(t, f, _p(v))
    return t


def mlp_block_desc(B, T, H, tok, ch, se_hidden, act, use_se, use_max, training, block_index, p, seed, step, precision=None,
                   step_dev=None):
    return L.MmxMlpBlockDesc(B, T, H, tok, ch, se_hidden, L.MMX_ACT[act], int(use_se), int(use_max), int(training),
                             block_index, L.MmxDropout(float(p), int(seed), int(step), _step_dev_ptr(step_dev)),
                             L.MMX_PREC[precision or _PRECISION])


class FusedMixerBlock(_Runner):
    """One MixerBlock as one fused kernel per direction.  The tcgen05 family runs each direction as two kernels (token half,
    channel half) and, when a training backward follows, can hand the token-half output x1 (+ SE gates) to it: one extra saved
    tile per block instead of re-running the token half forward (the save variant, ``saves``).

    ``dropout``: (seed, step, step_dev) of the masks, see ``dropout_source``."""

    def __init__(self, mb, B, device, need_backward, dropout):
        self.mb, self.B = mb, B
        self.seed, self.step, self.step_dev = dropout
        self.params = mb.kernel_params()
        self.w = mlp_block_table(self.params)
        self.out_shape = (B, mb.seq_len, mb.hidden_dim)
        self.saves = bool(need_backward and L.load().mmx_mlp_block_saves(C.byref(self._desc(True))))
        self.x1 = torch.empty(self.out_shape, device=device) if self.saves else None
        self.gate = torch.empty(B, mb.seq_len, device=device) if self.saves else None
        self.launches = (2, 2) if self.saves else (1, 1)

    def _desc(self, training):
        m = self.mb.meta(self.seed, self.step)
        return mlp_block_desc(self.B, self.mb.seq_len, self.mb.hidden_dim, *m[:6], training, *m[7:],
                              step_dev=self.step_dev if training else None)

    def forward(self, x, y, training):
        self.trained = training
        d = self._desc(training)
        if self.saves and training:
            _call("mmx_mlp_block_fwd_save", C.byref(d), C.byref(self.w), _p(x), _p(y), _p(self.x1), _p(self.gate), _stream())
        else:
            _call("mmx_mlp_block_fwd", C.byref(d), C.byref(self.w), _p(x), _p(y), _stream())

    def backward(self, x, dy, dx, grads):
        d, g = self._desc(self.trained), mlp_block_table(grads)
        if self.saves and self.trained:
            _call("mmx_mlp_block_bwd_saved", C.byref(d), C.byref(self.w), C.byref(g), _p(x), _p(self.x1), _p(self.gate), _p(dy), _p(dx),
                  _stream())
        else:
            _call("mmx_mlp_block_bwd", C.byref(d), C.byref(self.w), C.byref(g), _p(x), _p(dy), _p(dx), _stream())


class MlpBnBlock(_Runner):
    """The stage-kernel sequence of one MixerBlock whose MlpBlocks regularise with BatchNorm1d (regularization == -1,
    mlp_mixer.py:72-73, 88-94).

    Batch statistics are global over the batch, so the block is a chain of stage kernels (include/mmx.h, csrc/mmx_api_bnmlp.cu)
    with a reduction between them.  Token MLP: BatchNorm1d(hidden_dim) on [B,H,*]; channel MLP: BatchNorm1d(seq_len) on [B,T,*];
    reg1 after the activation, reg2 after fc2.  ``params``: MixerBlock.kernel_params() (14, SE weights may be None), then weight
    and bias of the four BatchNorm1d modules in execution order (token reg1, token reg2, channel reg1, channel reg2); their
    running statistics are updated in training mode exactly as nn.BatchNorm1d does."""
    saves = False
    launches = (16, 22)      # training: 2 LN + 4 fc + 4 x (stats, finalize) + 2 apply + 2 SE | 2 SE + 4 x (reduce, coef, apply) + 4 fc + 2 LN

    def __init__(self, mb, B, device, need_backward, dropout=None):
        e = _empty(device)
        T, H, tok, ch = mb.seq_len, mb.hidden_dim, mb.tokens_mlp_dim, mb.channels_mlp_dim
        self.mb = mb
        self.B, self.T, self.H, self.tok, self.ch = B, T, H, tok, ch
        self.bns = mb.bn_modules()
        self.params = mb.kernel_params() + [t for m in self.bns for t in (m.weight, m.bias)]
        self.act = L.MMX_ACT[mb.activation]
        self.se_hidden = mb.seq_len // mb.r_se if mb.use_se else 0
        self.use_max = int(mb.use_max_pooling)
        self.out_shape = (B, T, H)
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

    # channels / elements-per-channel of the four BatchNorm layers: (N, C, L)
    def _geo(self, i):
        B, T, H, tok, ch = self.B, self.T, self.H, self.tok, self.ch
        return [(B, H, tok), (B, H, T), (B, T, ch), (B, T, H)][i]

    def _bn_vectors(self, i, u, act, training):
        """per-channel vectors of BatchNorm layer i for the tensor u (pre-activation when act >= 0)."""
        N, Cn, Ln = self._geo(i)
        if training:
            _call("mmx_bn1d_stats", N, Cn, Ln, act, _p(u), _p(self.sums), _stream())
        return bn_vectors(self.bns[i], training, self.sums, N * Ln, self.bn[i])

    def forward(self, x, out, training):
        (ln1w, ln1b, tw1, tb1, tw2, tb2, ln2w, ln2b, cw1, cb1, cw2, cb2, s1, s2) = self.params[:14]
        B, T, H, tok, ch = self.B, self.T, self.H, self.tok, self.ch
        st = _stream()
        a, se_hidden, use_max = self.act, self.se_hidden, self.use_max
        self.trained = bool(training)
        # ---- token half: x1 = x + SE(BN(fc2(BN(act(fc1(LN1(x)^T)))))^T)
        _call("mmx_ln_fwd", B * T, H, T, _p(x), _p(ln1w), _p(ln1b), _p(self.nT), _p(self.st1), st)
        _call("mmx_linear_fwd", B * H, T, tok, _p(self.nT), _p(tw1), _p(tb1), _p(self.u1), st)
        bn = self._bn_vectors(0, self.u1, a, training)
        _call("mmx_bn1d_apply", B, H, tok, a, _p(self.u1), _p(bn), _p(self.g1), st)
        _call("mmx_linear_fwd", B * H, tok, T, _p(self.g1), _p(tw2), _p(tb2), _p(self.v1), st)
        bn = self._bn_vectors(1, self.v1, -1, training)
        _call("mmx_se_res_fwd", B, T, H, se_hidden, use_max, 1, 1, _p(x), _p(self.v1), _p(bn), _p(s1), _p(s2), _p(self.x1), st)
        # ---- channel half: out = x1 + SE(BN(fc2(BN(act(fc1(LN2(x1)))))))
        _call("mmx_ln_fwd", B * T, H, 0, _p(self.x1), _p(ln2w), _p(ln2b), _p(self.n2), _p(self.st2), st)
        _call("mmx_linear_fwd", B * T, H, ch, _p(self.n2), _p(cw1), _p(cb1), _p(self.u2), st)
        bn = self._bn_vectors(2, self.u2, a, training)
        _call("mmx_bn1d_apply", B, T, ch, a, _p(self.u2), _p(bn), _p(self.g2), st)
        _call("mmx_linear_fwd", B * T, ch, H, _p(self.g2), _p(cw2), _p(cb2), _p(self.v2), st)
        bn = self._bn_vectors(3, self.v2, -1, training)
        _call("mmx_se_res_fwd", B, T, H, se_hidden, use_max, 0, 0, _p(self.x1), _p(self.v2), _p(bn), _p(s1), _p(s2), _p(out), st)

    def _bn_backward(self, i, u, act, d, gw, gb):
        """d (gradient wrt the BatchNorm output, [N,C,L]) -> gradient wrt u, in place; gw / gb accumulated."""
        N, Cn, Ln = self._geo(i)
        st = _stream()
        _call("mmx_bn1d_bwd_reduce", N, Cn, Ln, act, _p(u), _p(self.bn[i]), _p(d), _p(self.sums), st)
        _call("mmx_bn_coef", _p(self.sums), Cn, float(N * Ln), _p(self.bn[i]), _p(self.coef), _p(gw), _p(gb), st)
        if not self.trained:               # eval mode: the statistics are constants, only the affine back-propagates
            self.coef[Cn:3 * Cn].zero_()
        _call("mmx_bn1d_bwd_apply", N, Cn, Ln, act, _p(u), _p(self.bn[i]), _p(self.coef), _p(d), _p(d), st)

    def backward(self, x, dout, dx, grads):
        """grads: tensors matching ``params`` (accumulated)."""
        (ln1w, ln1b, tw1, tb1, tw2, tb2, ln2w, ln2b, cw1, cb1, cw2, cb2, s1, s2) = self.params[:14]
        (g_ln1w, g_ln1b, g_tw1, g_tb1, g_tw2, g_tb2, g_ln2w, g_ln2b, g_cw1, g_cb1, g_cw2, g_cb2, g_s1, g_s2) = grads[:14]
        bn_grads = [grads[14 + 2 * i:16 + 2 * i] for i in range(4)]
        B, T, H, tok, ch = self.B, self.T, self.H, self.tok, self.ch
        st = _stream()
        a, se_hidden, use_max = self.act, self.se_hidden, self.use_max
        dA, dB, dC = self.dA, self.dB, self.dC
        # ---- channel half
        _call("mmx_se_res_bwd", B, T, H, se_hidden, use_max, 0, 0, _p(self.v2), _p(self.bn[3]), _p(s1), _p(s2), _p(dout),
              _p(g_s1), _p(g_s2), _p(dA), st)
        self._bn_backward(3, self.v2, -1, dA, *bn_grads[3])
        _call("mmx_linear_bwd", B * T, ch, H, _p(self.g2), _p(cw2), _p(dA), _p(g_cw2), _p(g_cb2), _p(dB), st)
        self._bn_backward(2, self.u2, a, dB, *bn_grads[2])
        _call("mmx_linear_bwd", B * T, H, ch, _p(self.n2), _p(cw1), _p(dB), _p(g_cw1), _p(g_cb1), _p(dA), st)
        _call("mmx_ln_bwd", B * T, H, 0, _p(self.x1), _p(self.st2), _p(ln2w), _p(dA), _p(dout), _p(dC), _p(g_ln2w), _p(g_ln2b), st)
        # ---- token half (dC = gradient wrt x1)
        _call("mmx_se_res_bwd", B, T, H, se_hidden, use_max, 1, 1, _p(self.v1), _p(self.bn[1]), _p(s1), _p(s2), _p(dC),
              _p(g_s1), _p(g_s2), _p(dA), st)
        self._bn_backward(1, self.v1, -1, dA, *bn_grads[1])
        _call("mmx_linear_bwd", B * H, tok, T, _p(self.g1), _p(tw2), _p(dA), _p(g_tw2), _p(g_tb2), _p(dB), st)
        self._bn_backward(0, self.u1, a, dB, *bn_grads[0])
        _call("mmx_linear_bwd", B * H, T, tok, _p(self.nT), _p(tw1), _p(dB), _p(g_tw1), _p(g_tb1), _p(dA), st)
        _call("mmx_ln_bwd", B * T, H, T, _p(x), _p(self.st1), _p(ln1w), _p(dA), _p(dC), _p(dx), _p(g_ln1w), _p(g_ln1b), st)


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


class MlpHead(_Runner):
    """MlpMixer head: LN -> conv_out -> fc_out (mlp_mixer.py:332-335)."""

    def __init__(self, model, B, device, need_backward):
        self.model = model
        self.params = [model.LN.weight, model.LN.bias, model.conv_out.weight, model.conv_out.bias, model.fc_out.weight, model.fc_out.bias]
        self.w = mlp_head_table(self.params)
        self.desc = L.MmxMlpHeadDesc(B, model.seq_len, model.pred_len, model.hidden_dim, model.num_classes)
        self.out_shape = (B, model.pred_len, model.num_classes)

    def forward(self, x, y, training):
        self.prec = L.MMX_PREC[self.model.precision or _PRECISION]
        _call("mmx_mlp_head_fwd_prec", C.byref(self.desc), C.byref(self.w), _p(x), _p(y), self.prec, _stream())

    def backward(self, x, dy, dx, grads):
        _call("mmx_mlp_head_bwd_prec", C.byref(self.desc), C.byref(self.w), C.byref(mlp_head_table(grads)), _p(x), _p(dy), _p(dx),
              self.prec, _stream())


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
# ConvMixer (conv_mixer_model.py, positional_encoder.py): encoder, ConvMixerBlock halves, SE tail, head
# ------------------------------------------------------------------------------------------------
def encoder_table(tensors):
    t = L.MmxEncoderParams()
    for f, v in zip(("freq", "w", "b", "wc", "bc"), tensors):
        setattr(t, f, _p(v))
    return t


class Encoder(_Runner):
    """PoseEncoder.forward (positional_encoder.py:79-97): harmonic embedding -> embed_mlp -> channelUpscaling.  Owns the
    embedding ``m`` [B*T, E] that the backward reads."""
    optional_dx = True

    def __init__(self, enc, B, device, need_backward):
        e = _empty(device)
        Hn = max(int(enc.n_harmonic_functions), 0)
        T, D, E, Cn = enc.in_nTP, enc.dimPosIn, enc.embed_mlp.out_features, enc.conv_nChan
        self.params = [enc.embed_mlp.weight, enc.embed_mlp.bias, enc.channelUpscaling.weight, enc.channelUpscaling.bias]
        self.w = encoder_table([enc.frequencies if Hn > 0 else None, *self.params])
        self.desc = L.MmxEncoderDesc(B, T, D, E, Cn, Hn)
        self.in_shape, self.out_shape = (B, T, D), (B, Cn, T, E)
        self.m = e(B * T, E)
        self.dm = e(B * T, E) if need_backward else None
        self.launches = (1, 2 if Hn == 0 else 3)

    def forward(self, x, y, training):
        _call("mmx_pose_encoder_fwd", C.byref(self.desc), C.byref(self.w), _p(x), _p(self.m), _p(y), _stream())

    def backward(self, x, dy, dx, grads):
        _call("mmx_pose_encoder_bwd", C.byref(self.desc), C.byref(self.w), C.byref(encoder_table([None, *grads])), _p(x), _p(self.m),
              _p(dy), _p(self.dm), _p(dx), _stream())


def conv_half_table(tensors, bn_aff=None):
    """tensors: (ln_w, ln_b, conv_w, conv_b, se_w1, se_w2) — the order of ``MmxConvHalfParams``; ``bn_aff``: optional
    eval-mode BatchNorm affine [scale | shift] (2C floats)."""
    t = L.MmxConvHalfParams()
    for f, v in zip(("ln_w", "ln_b", "conv_w", "conv_b", "se_w1", "se_w2"), tensors):
        setattr(t, f, _p(v))
    t.bn_aff = _p(bn_aff)
    return t


def conv_half_desc(B, Cn, T, E, kernel, pad, se_hidden, act, use_se, use_max, training, site, p, seed, step, step_dev=None):
    return L.MmxConvHalfDesc(B, Cn, T, E, kernel[0], kernel[1], pad[0], pad[1], se_hidden, L.MMX_ACT[act], int(use_se),
                             int(use_max), int(training), site, L.MmxDropout(float(p), int(seed), int(step), _step_dev_ptr(step_dev)))


def conv_prec(precision):
    """MMX_PREC_* of a ConvMixer convolution.  ``None`` is fp32: unlike the MlpMixer, the ConvMixer does not follow
    ``set_precision`` / MMX_PRECISION (ConvMixer runs under those settings have always been fp32 and stay bit for bit); it opts
    in through ``ConvMixer.set_precision("tf32")``."""
    return L.MMX_PREC[precision or "fp32"]


def conv_tc5_serves(B, Cn, T, E, meta):
    """True when precision "tf32" runs this half's convolutions on tcgen05 (mmx_conv2d_tc5_serves)."""
    return bool(L.load().mmx_conv2d_tc5_serves(C.byref(conv_half_desc(B, Cn, T, E, *meta))))


def conv_half_fits(B, Cn, T, E, meta):
    """True when the fused half kernels (forward and backward) serve this shape; else the stage-kernel chain runs."""
    desc = conv_half_desc(B, Cn, T, E, *meta)
    lib = L.load()
    return lib.mmx_conv_half_plan(C.byref(desc), 0, None, None) == 0 and lib.mmx_conv_half_plan(C.byref(desc), 1, None, None) == 0


class _Half(_Runner):
    """What both runners of one ConvMixerBlock half share: y = x + SE(reg(act(conv(LN(x))))) (conv_mixer_model.py:279-284 /
    :287-292).  ``params``: ConvMixerBlock.half_params(half), then the BatchNorm2d weight and bias when the half regularises
    with BatchNorm (regularization == -1).  ``dropout``: (seed, step, step_dev), see ``dropout_source``."""

    def __init__(self, mb, half, B, device, dropout):
        self.mb, self.half, self.B = mb, half, B
        self.seed, self.step, self.step_dev = dropout
        self.bnm = (mb.conv1 if half == 0 else mb.conv2).reg if mb.regularization == -1.0 else None
        self.params = mb.half_params(half) + ([self.bnm.weight, self.bnm.bias] if self.bnm is not None else [])
        self.C, self.T, self.E = mb.conv_nChan, mb.in_nTP, mb.dimPosEmb
        self.out_shape = (B, self.C, self.T, self.E)
        self.bn = torch.zeros(4 * self.C, dtype=torch.float32, device=device) if self.bnm is not None else None
        self.sums = torch.zeros(2 * self.C, dtype=torch.float64, device=device) if self.bnm is not None else None
        self.trained = True

    def _desc(self, training):
        m = self.mb.half_meta(self.half, self.seed, self.step)
        return conv_half_desc(self.B, self.C, self.T, self.E, *m[:6], training, *m[7:], step_dev=self.step_dev if training else None)


class ConvHalf(_Half):
    """One half as the fused kernels: one kernel per direction.  BatchNorm2d in training splits each direction at the batch
    reduction: statistics pass -> mmx_bn_finalize -> apply pass, and pass 1 (SE backward + batch sums) -> mmx_bn_coef -> pass 2
    (BN / conv / LN backward); the half owns ``z``, ``gd``, ``sums``, ``bn`` and ``coef``.  BatchNorm2d in eval is the constant
    affine [scale | shift] applied after the activation, and its parameters take no gradient."""

    def __init__(self, mb, half, B, device, need_backward, dropout):
        super().__init__(mb, half, B, device, dropout)
        self.w = conv_half_table(self.params[:6])
        if self.bnm is not None:
            e = _empty(device)
            self.w_eval = conv_half_table(self.params[:6], self.bn)
            self.z = e(self.out_shape)
            if need_backward:
                self.gd = e(B, self.T, 2)
                self.coef = torch.zeros(3 * self.C, dtype=torch.float32, device=device)

    def forward(self, x, y, training):
        self.trained = training
        d, st = self._desc(training), _stream()
        if self.bnm is None:
            _call("mmx_conv_half_fwd", C.byref(d), C.byref(self.w), _p(x), _p(y), st)
        elif training:
            _call("mmx_conv_half_bn_stats", C.byref(d), C.byref(self.w), _p(x), _p(self.z), _p(self.sums), st)
            bn_vectors(self.bnm, True, self.sums, self.B * self.T * self.E, self.bn)
            _call("mmx_conv_half_bn_apply", C.byref(d), C.byref(self.w), _p(self.bn), _p(x), _p(self.z), _p(y), st)
        else:
            bn_vectors(self.bnm, False, None, 0, self.bn)
            _call("mmx_conv_half_fwd", C.byref(d), C.byref(self.w_eval), _p(x), _p(y), st)

    def backward(self, x, dy, dx, grads):
        d, g, st = self._desc(self.trained), conv_half_table(grads[:6]), _stream()
        if self.bnm is None:
            _call("mmx_conv_half_bwd", C.byref(d), C.byref(self.w), C.byref(g), _p(x), _p(dy), _p(dx), st)
        elif self.trained:
            _call("mmx_conv_half_bn_bwd1", C.byref(d), C.byref(self.w), C.byref(g), _p(self.bn), _p(self.z), _p(dy), _p(self.gd),
                  _p(self.sums), st)
            _call("mmx_bn_coef", _p(self.sums), self.C, float(self.B * self.T * self.E), _p(self.bn), _p(self.coef), _p(grads[6]),
                  _p(grads[7]), st)
            _call("mmx_conv_half_bn_bwd2", C.byref(d), C.byref(self.w), C.byref(g), _p(self.bn), _p(self.coef), _p(x), _p(self.z),
                  _p(dy), _p(self.gd), _p(dx), st)
        else:
            _call("mmx_conv_half_bwd", C.byref(d), C.byref(self.w_eval), C.byref(g), _p(x), _p(dy), _p(dx), st)
            grads[6:] = [None, None]


class ConvHalfLarge(_Half):
    """One half that the fused kernels do not serve (mmx_conv_half_plan), or BatchNorm with the max squeeze, as a chain of
    stage kernels (include/mmx.h, csrc/mmx_api_conv_large.cu): LN -> conv2d -> [BatchNorm statistics] -> act / reg / SE /
    residual, intermediates in HBM.  The convolutions follow the block's precision, see ``conv_prec``."""

    def __init__(self, mb, half, B, device, need_backward, dropout):
        super().__init__(mb, half, B, device, dropout)
        e = _empty(device)
        B, Cn, T, E = self.out_shape
        self.prec = conv_prec(mb.precision)
        self.n, self.stats, self.z = e(B, Cn, T, E), e(B * Cn * T, 2), e(B, Cn, T, E)
        if need_backward:
            self.gd, self.dz, self.dn = e(B, T, 3), e(B, Cn, T, E), e(B, Cn, T, E)
            self.coef = e(3 * Cn) if self.bnm is not None else None
        self.launches = (5, 7) if self.bnm is not None else (3, 6)

    def forward(self, x, y, training):
        ln_w, ln_b, cw, cb, s1, s2 = self.params[:6]
        B, Cn, T, E = self.out_shape
        desc, st = self._desc(training), _stream()
        _call("mmx_ln_fwd", B * Cn * T, E, 0, _p(x), _p(ln_w), _p(ln_b), _p(self.n), _p(self.stats), st)
        _call("mmx_conv2d_large_fwd_prec", C.byref(desc), 0, _p(self.n), _p(cw), _p(cb), _p(self.z), self.prec, st)
        self.trained = bool(training)
        if self.bnm is not None and training:
            _call("mmx_bn1d_stats", B, Cn, T * E, desc.act, _p(self.z), _p(self.sums), st)
        if self.bnm is not None:
            bn_vectors(self.bnm, training, self.sums, B * T * E, self.bn)
        _call("mmx_conv_tail_fwd", C.byref(desc), _p(x), _p(self.z), _p(self.bn), _p(s1), _p(s2), _p(y), st)

    def backward(self, x, dy, dx, grads):
        ln_w, ln_b, cw, cb, s1, s2 = self.params[:6]
        g_ln_w, g_ln_b, g_cw, g_cb, g_s1, g_s2 = grads[:6]
        B, Cn, T, E = self.out_shape
        desc, st = self._desc(self.trained), _stream()
        bn = self.bn
        _call("mmx_conv_tail_bwd1", C.byref(desc), _p(self.z), _p(dy), _p(bn), _p(s1), _p(s2), _p(g_s1), _p(g_s2), _p(self.gd),
              _p(self.sums), st)
        if bn is not None:
            _call("mmx_bn_coef", _p(self.sums), Cn, float(B * T * E), _p(bn), _p(self.coef), _p(grads[6]), _p(grads[7]), st)
            if not self.trained:
                self.coef[Cn:3 * Cn].zero_()
        _call("mmx_conv_tail_bwd2", C.byref(desc), _p(self.z), _p(dy), _p(self.gd), _p(bn), _p(self.coef), _p(self.dz), st)
        _call("mmx_conv2d_large_wgrad_prec", C.byref(desc), _p(self.dz), _p(self.n), _p(g_cw), _p(g_cb), self.prec, st)
        _call("mmx_conv2d_large_fwd_prec", C.byref(desc), 1, _p(self.dz), _p(cw), None, _p(self.dn), self.prec, st)
        _call("mmx_ln_bwd", B * Cn * T, E, 0, _p(x), _p(self.stats), _p(ln_w), _p(self.dn), _p(dy), _p(dx), _p(g_ln_w), _p(g_ln_b), st)


class SeTail(_Runner):
    """mode_conv='once': y = x + se(x), or 2x without SE (conv_mixer_model.py:259-263,287-292)."""

    def __init__(self, mb, B, device, need_backward):
        self.mb = mb
        self.params = mb.se_weights()
        self.out_shape = (B, mb.conv_nChan, mb.in_nTP, mb.dimPosEmb)
        self.args = (*self.out_shape, mb.in_nTP // mb.r_se if mb.use_se else 0, int(mb.use_se), int(mb.use_max_pooling))

    def forward(self, x, y, training):
        s1, s2 = self.params
        _call("mmx_se_tail_fwd", *self.args, _p(s1), _p(s2), _p(x), _p(y), _stream())

    def backward(self, x, dy, dx, grads):
        s1, s2 = self.params
        _call("mmx_se_tail_bwd", *self.args, _p(s1), _p(s2), _p(grads[0]), _p(grads[1]), _p(x), _p(dy), _p(dx), _stream())


def conv_head_table(tensors):
    t = L.MmxConvHeadParams()
    for f, v in zip(("ln_w", "ln_b", "wt", "bt", "wp", "bp", "wf", "bf"), tensors):
        setattr(t, f, _p(v))
    return t


class ConvHead(_Runner):
    """LN -> conv_out -> project_channels -> GELU -> fc_out (conv_mixer_model.py:455-463)."""

    def __init__(self, model, B, device, need_backward):
        self.params = model.head_params()
        self.w = conv_head_table(self.params)
        self.desc = L.MmxConvHeadDesc(B, model.conv_nChan, model.in_nTP, model.out_nTP, model.dimPosEmb, model.dimPosOut)
        self.out_shape = (B, model.out_nTP, model.dimPosOut)

    def forward(self, x, y, training):
        _call("mmx_conv_head_fwd", C.byref(self.desc), C.byref(self.w), _p(x), _p(y), _stream())

    def backward(self, x, dy, dx, grads):
        _call("mmx_conv_head_bwd", C.byref(self.desc), C.byref(self.w), C.byref(conv_head_table(grads)), _p(x), _p(dy), _p(dx), _stream())


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
