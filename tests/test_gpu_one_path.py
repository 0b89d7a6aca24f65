"""GPU (-m gpu): the autograd path and TrainStep launch the same kernel sequence.

Both host paths build their layers from ``model.runners`` (functional.py).  For every runner branch this records the C ABI
calls, by wrapping the library object ``_lib.load()`` returns, of
  (a) one eager ``TrainStep`` step, and ``TrainStep.predict``;
  (b) ``model(x)`` -> ``mpjpe_error`` -> ``backward`` -> ``FusedAdam.step``, and ``model(x)`` in eval under ``no_grad``;
and requires the same entry points with the same descriptor fields and scalar arguments (pointers compared only for being
null or not, the dropout step source left out), and the same gradient buckets and predictions up to the order in which kernels sum with atomics.
"""
import ctypes as C

import pytest
import torch

from motionmixerconv_b200 import _lib as L
from tests.synthetic import synthetic_pose_windows

MLP = dict(num_classes=66, num_blocks=2, hidden_dim=50, tokens_mlp_dim=20, channels_mlp_dim=50, seq_len=10, pred_len=10,
           activation="mish", regularization=0, input_size=66, r_se=8, use_se=True)
CONV = dict(num_blocks=2, dimPosIn=33, dimPosEmb=48, dimPosOut=33, in_nTP=10, out_nTP=10, conv_nChan=4, conv1_kernel_shape=(3, 3),
            mode_conv="twice", activation="mish", regularization=0, use_se=True, r_se=4, encoder_n_harmonic_functions=4,
            encoder_omega0=0.1)
LARGE = dict(num_blocks=1, dimPosIn=33, dimPosEmb=192, dimPosOut=33, in_nTP=10, out_nTP=10, conv_nChan=8, activation="mish",
             use_se=True, r_se=8, encoder_n_harmonic_functions=0, encoder_omega0=0, conv1_kernel_shape=(5, 9), mode_conv="twice",
             regularization=0)

# name -> (family, config, precision, MMX_CONV_FORCE_LARGE, the runner classes the blocks must take)
CASES = {
    "mlp_fp32": ("mlp", MLP, "fp32", False, {"FusedMixerBlock"}),
    "mlp_tf32_saves": ("mlp", MLP, "tf32", False, {"FusedMixerBlock"}),
    "mlp_bn": ("mlp", dict(MLP, regularization=-1.0), None, False, {"MlpBnBlock"}),
    "conv_fused": ("conv", CONV, None, False, {"ConvHalf"}),
    "conv_once_se_tail": ("conv", dict(CONV, mode_conv="once"), None, False, {"ConvHalf", "SeTail"}),
    "conv_fused_bn": ("conv", dict(CONV, regularization=-1.0), None, False, {"ConvHalf"}),
    "conv_chain_forced": ("conv", CONV, None, True, {"ConvHalfLarge"}),
    "conv_chain_bn_max": ("conv", dict(CONV, regularization=-1.0, use_max_pooling=True), None, False, {"ConvHalfLarge"}),
    "conv_chain_tf32": ("conv", LARGE, "tf32", False, {"ConvHalfLarge"}),
}
B = 24
# queries the routing asks once per runner or module, not kernel launches
QUERIES = {"mmx_mlp_block_saves", "mmx_conv_half_plan", "mmx_conv2d_tc5_serves", "mmx_tc5_abort_count", "mmx_last_error"}


class _Recorder:
    """Stands in for the loaded library: every mmx_* call is recorded as (name, canonical arguments) while ``calls`` is a list."""

    def __init__(self, lib):
        self.lib, self.calls = lib, None

    def __getattr__(self, name):
        fn = getattr(self.lib, name)
        if name not in L.SIGNATURES or name in QUERIES:
            return fn

        def call(*args):
            if self.calls is not None:
                self.calls.append((name, tuple(_canon(a, t) for a, t in zip(args, L.SIGNATURES[name][1]))))
            return fn(*args)
        return call


def _canon(arg, argtype):
    if argtype is C.c_void_p:
        return "null" if (arg.value if isinstance(arg, C.c_void_p) else arg) is None else "ptr"
    if isinstance(argtype, type) and issubclass(argtype, C._Pointer) and issubclass(argtype._type_, C.Structure):
        return _struct(arg._obj)
    return arg


def _struct(s):
    out = []
    for f, t in s._fields_:
        v = getattr(s, f)
        if t is C.c_void_p:
            out.append((f, "null" if v is None else "ptr"))
        elif t is L.MmxDropout:          # the step source (host step, device counter) differs by design
            out.append((f, (round(v.p, 6), v.seed if v.p > 0 else None)))
        else:
            out.append((f, v))
    return tuple(out)


@pytest.fixture
def recorder(monkeypatch):
    rec = _Recorder(L.load())
    monkeypatch.setattr(L, "_lib", rec)
    return rec


def _model(family, cfg, precision):
    from motionmixerconv_b200.conv_mixer_model import ConvMixer
    from motionmixerconv_b200.mlp_mixer import MlpMixer
    torch.manual_seed(7)
    m = (MlpMixer if family == "mlp" else ConvMixer)(**cfg).cuda().train()
    return m.set_precision(precision) if precision else m


def _data(family, cfg):
    T, To, D = (cfg["seq_len"], cfg["pred_len"], cfg["input_size"]) if family == "mlp" else (cfg["in_nTP"], cfg["out_nTP"], cfg["dimPosIn"])
    x, gt = synthetic_pose_windows(B, T, To, D, scale="h36m", seed=5)
    return torch.from_numpy(x).cuda(), torch.from_numpy(gt).cuda()


def _record(rec, fn):
    rec.calls = []
    out = fn()
    torch.cuda.synchronize()
    calls, rec.calls = rec.calls, None
    return calls, out


def _same_calls(a, b):
    for i, (ca, cb) in enumerate(zip(a, b)):
        assert ca == cb, "call %d differs:\n  TrainStep %s\n  autograd  %s" % (i, ca, cb)
    assert len(a) == len(b), ([c[0] for c in a[len(b):]], [c[0] for c in b[len(a):]])


@pytest.mark.gpu
@pytest.mark.parametrize("case", sorted(CASES))
def test_trainstep_and_autograd_launch_the_same_kernels(case, recorder, monkeypatch):
    from motionmixerconv_b200.functional import mpjpe_error
    from motionmixerconv_b200.train import FusedAdam, TrainStep
    family, cfg, precision, force_large, kinds = CASES[case]
    if force_large:
        monkeypatch.setenv("MMX_CONV_FORCE_LARGE", "1")
    x, gt = _data(family, cfg)
    m_ts, m_ag = _model(family, cfg, precision), _model(family, cfg, precision)
    ts = TrainStep(m_ts, lr=1e-3, weight_decay=1e-5, use_cuda_graph=False)
    opt = FusedAdam(m_ag.parameters(), lr=1e-3, weight_decay=1e-5)

    # eval: TrainStep.predict against model(x) under no_grad
    pa, pred_a = _record(recorder, lambda: ts.predict(x).clone())
    m_ag.eval()
    with torch.no_grad():
        pb, pred_b = _record(recorder, lambda: m_ag(x))
    m_ag.train()
    _same_calls(pa, pb)
    if family == "mlp":
        assert torch.equal(pred_a, pred_b)
    else:           # the encoder's split-K partial sums combine in any order (the bar of tests/test_gpu_rollout.py)
        assert (pred_a - pred_b).abs().max().item() <= 2e-6 * pred_b.abs().max().item()

    blocks = ts.plan.runs[1:-1]
    assert {type(r).__name__ for r in blocks} == kinds
    if case == "mlp_tf32_saves":
        assert all(ts.plan.saves)
    if case == "conv_chain_tf32":
        assert all(mb.uses_tc5_conv(h, B) for mb in m_ts.Mixer_Block for h in (0, 1))

    # one training step
    sa, loss_a = _record(recorder, lambda: float(ts.step(x, gt)))

    def autograd_step():
        opt.zero_grad(set_to_none=True)
        loss = mpjpe_error(m_ag(x), gt)
        loss.backward()
        opt.step()
        return float(loss)
    sb, loss_b = _record(recorder, autograd_step)
    _same_calls(sa, sb)
    assert loss_a == pytest.approx(loss_b, rel=1e-6 if family == "mlp" else 1e-5)
    ga, gb = ts.flat.g, opt.flat(0).g
    assert ga.shape == gb.shape
    # weight gradients summed by atomics from several CTAs differ in the order of the sum (the bar of tests/test_gpu_rollout.py)
    scale = ga.abs().max().item()
    for name, off, n, _ in ts._named_flat():
        assert (ga[off:off + n] - gb[off:off + n]).abs().max().item() <= 2e-5 * scale, name
    for (k, va), vb in zip(m_ts.named_buffers(), m_ag.buffers()):       # BatchNorm running statistics
        assert torch.allclose(va, vb, rtol=1e-5, atol=1e-6), k


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["conv_fused_bn", "conv_chain_bn_max"])
def test_batchnorm_momentum_follows_the_module(case):
    """Running statistics after one training forward from (mean 0, var 1): nn.BatchNorm2d gives momentum * batch mean and
    (1 - momentum) + momentum * unbiased batch variance, so momentum 0.3 moves them three times as far as momentum 0.1."""
    family, cfg, precision, _, kinds = CASES[case]
    x, _ = _data(family, cfg)
    stats = {}
    for momentum in (0.1, 0.3):
        model = _model(family, cfg, precision)
        bns = [m for m in model.modules() if isinstance(m, torch.nn.BatchNorm2d)]
        for m in bns:
            m.momentum = momentum
        assert {type(r).__name__ for r in list(model.runners(B, x.device, False))[1:-1]} == kinds
        with torch.no_grad():
            model(x)
        stats[momentum] = [(m.running_mean.clone(), m.running_var.clone()) for m in bns]
    for (rm1, rv1), (rm3, rv3) in zip(stats[0.1], stats[0.3]):
        mean, var = rm1 / 0.1, (rv1 - 0.9) / 0.1
        assert torch.allclose(rm3, 0.3 * mean, rtol=1e-5, atol=1e-6)
        assert torch.allclose(rv3, 0.7 + 0.3 * var, rtol=1e-5, atol=1e-5)
