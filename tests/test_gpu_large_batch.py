"""Large batches against the oracle: every channel-half plan of the tcgen05 MixerBlock family with several tiles per CTA, the
default plan policy at the large-batch sweep's sizes (16K - 256K sequences, tools/sweep.py), dropout and the TrainStep graph
at the batch where the backward switches plans, and the FP32 / ConvMixer kernels at ~65K sequences.

Two constructions keep the fp64 oracle cheap at these sizes and still see a single wrong tile:

  * replicated batch: x[i] = base[i % P] with P = 1031 distinct sequences (prime: no common factor with a tile of 2 - 20
    sequences or a CTA count).  Without BatchNorm and dropout sequences are independent, so EVERY row of the prediction and
    of dx is checked against the oracle run on the base set, and the mean-loss parameter gradients equal the base-set
    gradients with dpred row p weighted by count_p * P / B (exact).
  * sparse upstream gradient: pred.backward(dpred) with dpred nonzero on ~64 sequences spread over the batch.  Each of them
    carries ~1/64 of every weight gradient, so a tile lost, counted twice or read at the wrong offset moves a gradient by
    percent, far beyond the 2e-3 bar, where at B = 16K a whole-batch comparison would move by 7e-4.  dx must be exactly 0
    outside the selected sequences (the backward is linear in dy): a tile that reads another tile's dy shows up there.

test_replicated_and_sparse_constructions_are_exact checks both constructions on the CPU with the fp64 oracle.
"""
import collections
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import mixer_np as O
from oracle import mixer_torch as MT
from tests import masks_np as MK
from tests.golden_util import check_close, grad_scale
from tests.synthetic import synthetic_pose_windows

TOL = 2e-3          # reduced-precision (tcgen05) mode, every tensor
TOL_FP32 = 1e-5     # FP32 kernels
P = 1031            # distinct sequences of the replicated batch
N_SPARSE = 64       # sequences that carry the sparse upstream gradient
CHUNK = 16384       # rows per chunk of the on-device row comparison

Rep = collections.namedtuple("Rep", "pred loss grads dx")


def mlp_cfg(H, ch=None, **kw):
    """The large-batch sweep's MlpMixer (tools/sweep.py) without dropout."""
    c = dict(num_classes=66, num_blocks=4, hidden_dim=H, tokens_mlp_dim=20, channels_mlp_dim=H if ch is None else ch, seq_len=10,
             pred_len=10, activation="mish", regularization=0, input_size=66, r_se=8, use_se=True)
    c.update(kw)
    return c


def conv_cfg(E):
    """The large-batch sweep's ConvMixer (tools/sweep.py) without dropout."""
    return dict(num_blocks=4, dimPosIn=66, dimPosEmb=E, dimPosOut=66, in_nTP=10, out_nTP=25, conv_nChan=1, conv1_kernel_shape=(1, 3),
                conv1_stride=(1, 1), conv1_padding=(0, 1), mode_conv="twice", activation="mish", regularization=0, use_se=True, r_se=8,
                encoder_n_harmonic_functions=0, encoder_omega0=0)


# ------------------------------------------------------------------------------------------ the two oracle constructions
def replicated_oracle(oracle, xb, gtb, B):
    """Oracle of the batch x[i] = xb[i % P], gt[i] = gtb[i % P] (i < B) under the mean MPJPE, run on the P base sequences only.
    ``oracle``: a fresh MlpMixerOracle / ConvMixerOracle.  pred[p] and dx[p] are what row i = p (mod P) of the batch must
    give; grads and loss are those of the whole batch."""
    n = len(xb)
    count = np.bincount(np.arange(B) % n, minlength=n).astype(oracle.dtype)
    pred = oracle.forward(xb, training=True)
    gt = gtb.astype(oracle.dtype)
    nrm = np.sqrt(((gt - pred).reshape(n, -1, 3) ** 2).sum(-1))                 # [P, joints per sequence]
    loss = float((count * nrm.sum(1)).sum() / (B * nrm.shape[1]))
    _, dp = O.mpjpe(pred, gt)                                                  # row p: d(mean over the P base rows)
    w = (count * n / B)[:, None, None]                                         # -> d(mean over B rows), summed over p's copies
    grads, dxw = oracle.backward(dp * w)
    return Rep(pred, loss, grads, dxw / count[:, None, None])


def sparse_rows(B, seed, n=N_SPARSE):
    """The first and the last sequence and a seeded sample spread over the batch."""
    rng = np.random.default_rng(seed)
    mid = rng.choice(np.arange(1, B - 1), size=min(n, B) - 2, replace=False)
    return np.unique(np.concatenate([[0, B - 1], mid]))


def sparse_dpred(shape, q, seed):
    """Upstream gradient rows for the sequences q (fp32, of the magnitude the mean loss gives them)."""
    rng = np.random.default_rng(seed)
    return (rng.standard_normal((len(q),) + tuple(shape[1:])) / (len(q) * shape[1] * shape[2] / 3)).astype(np.float32)


def sparse_oracle(oracle, xq, dq):
    """Parameter gradients and dx of the sequences xq alone under the upstream gradient rows dq."""
    oracle.forward(xq, training=True)
    return oracle.backward(dq)


def test_replicated_and_sparse_constructions_are_exact():
    """CPU, fp64 oracle, tiny P: (1) the replicated-batch oracle equals the oracle of the whole replicated batch; (2) with a
    sparse dpred the whole batch's gradients equal those of the selected sequences alone, and dx is exactly 0 elsewhere."""
    cfg = mlp_cfg(12, 10, num_blocks=2)
    params = {k: v.numpy() for k, v in MT.random_params("mlp", cfg, seed=5).items()}
    n, B = 7, 3 * 7 + 4
    xb, gtb = synthetic_pose_windows(n, 10, 10, 66, scale="amass", seed=2)
    x, gt = xb[np.arange(B) % n], gtb[np.arange(B) % n]

    full = O.MlpMixerOracle(cfg, params, dtype=np.float64)
    pred = full.forward(x, training=True)
    loss, dp = O.mpjpe(pred, gt.astype(np.float64))
    grads, dx = full.backward(dp)
    rep = replicated_oracle(O.MlpMixerOracle(cfg, params, dtype=np.float64), xb, gtb, B)

    def close(a, b, scale=0.0):       # scale: the gradient scale (some bias gradients are 0 up to fp64 rounding)
        return float(np.abs(a - b).max()) <= 1e-12 * float(np.abs(b).max()) + 1e-14 * scale

    assert close(rep.pred[np.arange(B) % n], pred)
    assert abs(rep.loss - float(loss)) < 1e-12 * float(loss)
    assert close(rep.dx[np.arange(B) % n], dx)
    for k, g in grads.items():
        assert close(rep.grads[k], g, grad_scale(grads)), k

    q = sparse_rows(B, seed=1, n=5)
    assert q[0] == 0 and q[-1] == B - 1 and len(q) == 5
    dq = sparse_dpred(pred.shape, q, seed=1).astype(np.float64)
    dpred = np.zeros_like(pred)
    dpred[q] = dq
    grads, dx = full.backward(dpred)
    gq, dxq = sparse_oracle(O.MlpMixerOracle(cfg, params, dtype=np.float64), x[q], dq)
    for k, g in grads.items():
        assert close(gq[k], g, grad_scale(grads)), k
    assert close(dxq, dx[q])
    outside = np.ones(B, bool)
    outside[q] = False
    assert not dx[outside].any()


# ------------------------------------------------------------------------------------------ GPU side
def _mlp_module(cfg, seed):
    from motionmixerconv_b200.mlp_mixer import MlpMixer
    torch.manual_seed(seed)
    return MlpMixer(**cfg)


def _mlp(cfg, seed=3, precision="tf32"):
    m = _mlp_module(cfg, seed)
    params = {k: v.detach().numpy().copy() for k, v in m.state_dict().items()}
    return m.cuda().set_precision(precision).train(), params


def _conv(cfg, seed=3):
    from motionmixerconv_b200.conv_mixer_model import ConvMixer
    torch.manual_seed(seed)
    m = ConvMixer(**cfg)
    params = {k: v.detach().numpy().copy() for k, v in m.state_dict().items()}
    return m.cuda().train(), params


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _assert_healthy():
    from motionmixerconv_b200 import _lib as L
    assert L.load().mmx_tc5_abort_count() == 0            # no pipeline wait of the tcgen05 family ever timed out


def _assert_tc5_serves(model, B):
    from motionmixerconv_b200 import _lib as L
    from motionmixerconv_b200 import functional as F_
    mb = model.Mixer_Block[0]
    desc = F_.mlp_block_desc(B, mb.seq_len, mb.hidden_dim, *mb.meta())
    assert L.load().mmx_mlp_block_saves(C.byref(desc)) == 1       # else a silent FP32 fall-back would pass these tests


def check_rows(name, got, want, truth=None, rtol=TOL, atol=0.0):
    """Row i of the CUDA tensor ``got`` [B, ...] must equal row i % P of ``want`` [P, ...].  The difference is taken on the
    device, chunk by chunk; check_close then gets the P base rows plus the worst row of the batch (against ``want``, and
    against ``truth`` for the noise clause), so its scale, noise and worst error are exactly those of all B rows."""
    n, B, dev = len(want), got.shape[0], got.device
    rows = set()
    for ref in [want] if truth is None else [want, truth]:
        r = torch.from_numpy(np.ascontiguousarray(ref, dtype=np.float64)).to(dev)
        err = torch.empty(B, dtype=torch.float64, device=dev)
        for s in range(0, B, CHUNK):
            e = min(B, s + CHUNK)
            err[s:e] = (got[s:e].double() - r[torch.arange(s, e, device=dev) % n]).abs().flatten(1).amax(1)
        assert bool(torch.isfinite(err).all()), "%s: non-finite values" % name
        rows.add(int(err.argmax()))
    sel = np.concatenate([np.arange(n), sorted(rows)])
    g = got[torch.from_numpy(sel).to(dev)].cpu().numpy()
    return check_close(name, g, want[sel % n], None if truth is None else truth[sel % n], rtol=rtol, atol=atol)


def _replicate(a, B):
    ad = torch.from_numpy(a).cuda()
    return ad[torch.arange(B, device="cuda") % len(a)].contiguous()


def _check_replicated(model, oracles, xb, gtb, B, tol, floor_k, dx_atol_k=0.0, grad_atol=None):
    """Full batch x[i] = xb[i % P] through autograd + mean MPJPE against the replicated-batch oracle.  ``oracles``: fresh
    oracles, the first is compared with (the second, if any, is the fp64 truth of the noise clause)."""
    from motionmixerconv_b200.functional import mpjpe_error
    reps = [replicated_oracle(o, xb, gtb, B) for o in oracles]
    want, truth = reps[0], (reps[1] if len(reps) > 1 else None)
    model.zero_grad()
    x = _replicate(xb, B).requires_grad_(True)
    pred = model(x)
    loss = mpjpe_error(pred, _replicate(gtb, B))
    loss.backward()
    torch.cuda.synchronize()
    check_rows("pred", pred.detach(), want.pred, None if truth is None else truth.pred, rtol=tol)
    ref_loss = (truth or want).loss
    assert abs(float(loss.detach()) - ref_loss) <= tol * abs(ref_loss), (float(loss.detach()), ref_loss)
    floor = floor_k * grad_scale(want.grads)
    grads = {k: p.grad.detach().cpu().numpy() for k, p in model.named_parameters()}
    for k in O.trainable_keys(want.grads):
        if ".se2." in k:
            continue
        atol = floor * (grad_atol(k) if grad_atol else 1.0)
        check_close("grad " + k, grads[k], want.grads[k], None if truth is None else truth.grads[k], rtol=tol, atol=atol)
    check_rows("dx", x.grad, want.dx, None if truth is None else truth.dx, rtol=tol, atol=dx_atol_k * float(np.abs(want.dx).max()))


def _check_sparse(model, oracles, xb, B, tol, floor_k, seed=11):
    """Forward of the whole batch, backward of a dpred that is nonzero on ~64 sequences only.  ``oracles`` as in
    _check_replicated."""
    q = sparse_rows(B, seed)
    model.zero_grad()
    x = _replicate(xb, B).requires_grad_(True)
    pred = model(x)
    dq = sparse_dpred(pred.shape, q, seed)
    dpred = torch.zeros_like(pred)
    qd = torch.from_numpy(q).cuda()
    dpred[qd] = torch.from_numpy(dq).cuda()
    pred.backward(dpred)
    torch.cuda.synchronize()
    res = [sparse_oracle(o, xb[q % len(xb)], dq.astype(o.dtype)) for o in oracles]
    (gq, dxq), (gt_, dxt) = res[0], (res[1] if len(res) > 1 else (collections.defaultdict(lambda: None), None))
    floor = floor_k * grad_scale(gq)
    grads = {k: p.grad.detach().cpu().numpy() for k, p in model.named_parameters()}
    for k in O.trainable_keys(gq):
        if ".se2." in k:
            continue
        check_close("sparse grad " + k, grads[k], gq[k], gt_[k], rtol=tol, atol=floor)
    check_close("sparse dx", x.grad[qd].cpu().numpy(), dxq, dxt, rtol=tol)
    outside = torch.ones(B, dtype=torch.bool, device="cuda")
    outside[qd] = False
    leaked = torch.nonzero(outside & (x.grad.flatten(1) != 0).any(1))
    assert leaked.numel() == 0, "dx nonzero outside the sequences that carry dpred, first at %s" % leaked[:8].flatten().tolist()


def _check_tc5(cfg, B, seed=3):
    model, params = _mlp(cfg, seed)
    _assert_tc5_serves(model, B)
    xb, gtb = synthetic_pose_windows(P, cfg["seq_len"], cfg["pred_len"], cfg["input_size"], scale="amass", seed=seed + 40)
    _check_replicated(model, [O.MlpMixerOracle(cfg, params, dtype=np.float64)], xb, gtb, B, TOL, 0.01 * TOL)
    _assert_healthy()
    _check_sparse(model, [O.MlpMixerOracle(cfg, params, dtype=np.float64)], xb, B, TOL, 0.01 * TOL)
    _assert_healthy()


# ------------------------------------------------------------------------------------------ every channel-half plan, >= 3 tiles per CTA
# name: (H, ch, MMX_CHAN_STREAMED).  The knob (read on every call) forces the plan where H, ch <= 64 and ch is even:
# 0 = resident weights (operand width 64, or 80 when max(H, ch) + 1 > 64), 3 = streamed weights at width 64, forward and
# backward (two CTAs per SM).  Wider shapes have one plan each: resident at width 80 (max(H, ch) < 80), streamed at 128.
PLANS = {
    "h50_resident": (50, 50, 0),          # width 64, 2-float row loads (H % 4 != 0)
    "h50_streamed": (50, 50, 3),
    "h48_ch40_resident": (48, 40, 0),     # width 64, 4-float row loads
    "h48_ch40_streamed": (48, 40, 3),
    "h64_streamed": (64, 64, 3),          # width 64 holds H = 64 only without the resident plan's ones column
    "h64_resident_w80": (64, 64, 0),
    "h72_resident_w80": (72, 72, None),   # width 80, 4-float row loads
    "h128_streamed_w128": (128, 128, None),
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(PLANS))
def test_channel_plan_with_several_tiles_per_cta(name, monkeypatch):
    """B such that every CTA of the channel half runs >= 3 tiles of 12 sequences (at most 2 CTAs per SM in every plan) and the
    last tile is ragged: the weight-slot cycle and its mbarrier phases, dW accumulated in TMEM across tiles, the next-tile
    prefetch."""
    H, ch, streamed = PLANS[name]
    if streamed is None:
        monkeypatch.delenv("MMX_CHAN_STREAMED", raising=False)
    else:
        monkeypatch.setenv("MMX_CHAN_STREAMED", str(streamed))
    sms = _sms()
    B = 3 * 2 * sms * 12 + 5
    assert B > 3 * 2 * sms * 12 and B % 12 != 0
    _check_tc5(mlp_cfg(H, ch), B)


# ------------------------------------------------------------------------------------------ the default policy at the sweep's sizes
def _threshold_batch(sms):
    """Smallest batch whose backward has 8 x SMs channel tiles (12 sequences each): where the default policy sends the
    H, ch <= 63 backward to the streamed plan."""
    B = 12 * 8 * sms - 11
    assert (B + 11) // 12 >= 8 * sms > (B - 1 + 11) // 12
    return B


SWEEP_B = {"threshold": None, "65K": 65537, "262K": 262905}


@pytest.mark.gpu
@pytest.mark.parametrize("H", [50, 64, 128])
@pytest.mark.parametrize("size", list(SWEEP_B))
def test_default_policy_at_sweep_batch_sizes(H, size, monkeypatch):
    monkeypatch.delenv("MMX_CHAN_STREAMED", raising=False)
    B = SWEEP_B[size] or _threshold_batch(_sms())
    _check_tc5(mlp_cfg(H), B)


@pytest.mark.gpu
def test_fp32_kernels_at_65k():
    """FP32 MixerBlock kernels (warp per sequence pair, contended shared-memory accumulators) at 65K sequences."""
    cfg = mlp_cfg(50)
    B = SWEEP_B["65K"]
    model, params = _mlp(cfg, seed=4, precision="fp32")
    xb, gtb = synthetic_pose_windows(P, 10, 10, 66, scale="amass", seed=44)
    _check_replicated(model, [O.MlpMixerOracle(cfg, params, dtype=dt) for dt in (np.float32, np.float64)], xb, gtb, B,
                      TOL_FP32, 1e-6, dx_atol_k=1e-6)
    _check_sparse(model, [O.MlpMixerOracle(cfg, params, dtype=dt) for dt in (np.float32, np.float64)], xb, B, TOL_FP32, 1e-6)


@pytest.mark.gpu
def test_convmixer_at_65k():
    """Fused FP32 ConvMixer kernels, the sweep's E = 256 model, at 65K sequences."""
    cfg = conv_cfg(256)
    B = SWEEP_B["65K"]
    model, params = _conv(cfg, seed=4)
    xb, gtb = synthetic_pose_windows(P, 10, 25, 66, scale="amass", seed=45)
    _check_replicated(model, [O.ConvMixerOracle(cfg, params, dtype=dt) for dt in (np.float32, np.float64)], xb, gtb, B,
                      TOL_FP32, 5e-6, dx_atol_k=1e-6, grad_atol=lambda k: 50 if k == "encoder.channelUpscaling.bias" else 1)
    _check_sparse(model, [O.ConvMixerOracle(cfg, params, dtype=dt) for dt in (np.float32, np.float64)], xb, B, TOL_FP32, 5e-6)


# ------------------------------------------------------------------------------------------ dropout and TrainStep at the threshold batch
@pytest.mark.gpu
def test_dropout_at_the_threshold_batch(monkeypatch):
    """Dropout 0.1 (the sweep's setting) where the backward switches to the streamed plan: the full fp64 oracle with the masks
    the kernels draw.  Masks are per sequence, so this one is not a replicated batch."""
    from tests.test_gpu_mlp_tc5 import _compare, _oracle, _run
    monkeypatch.delenv("MMX_CHAN_STREAMED", raising=False)
    cfg = mlp_cfg(50, regularization=0.1)
    B = _threshold_batch(_sms())
    x, gt = synthetic_pose_windows(B, 10, 10, 66, scale="amass", seed=23)
    model, params = _mlp(cfg, seed=4321)
    torch.manual_seed(4321)                                 # the blocks draw their dropout seed from torch.initial_seed()
    _assert_tc5_serves(model, B)
    got = _run(model, x, gt)
    _compare(*got, _oracle(cfg, params, x, gt, masks=MK.mlp_tc5_masks(cfg, B, 4321, step=0)))
    _assert_healthy()


@pytest.mark.gpu
def test_train_step_at_the_threshold_batch(monkeypatch):
    """TrainStep drives the kernels through its own plan and CUDA graph (what the sweep times), not through autograd: one
    step on a replicated batch, the loss and every gradient of the flat buffer against the replicated-batch oracle."""
    from motionmixerconv_b200.train import TrainStep
    monkeypatch.delenv("MMX_CHAN_STREAMED", raising=False)
    cfg = mlp_cfg(50)
    B = _threshold_batch(_sms())
    model, params = _mlp(cfg, seed=6)
    xb, gtb = synthetic_pose_windows(P, 10, 10, 66, scale="amass", seed=46)
    want = replicated_oracle(O.MlpMixerOracle(cfg, params, dtype=np.float64), xb, gtb, B)
    ts = TrainStep(model, lr=1e-3, weight_decay=1e-5)
    loss = float(ts.step(_replicate(xb, B), _replicate(gtb, B)))
    torch.cuda.synchronize()
    assert all(ts.plan.saves)                                # the tcgen05 family served every block
    assert abs(loss - want.loss) <= TOL * abs(want.loss), (loss, want.loss)
    floor = 0.01 * TOL * grad_scale(want.grads)
    named = ts._named_flat()
    assert sorted(n for n, *_ in named) == sorted(O.trainable_keys(want.grads))
    for n, off, k, shape in named:
        check_close("grad " + n, ts.flat.g[off:off + k].view(shape).cpu().numpy(), want.grads[n], rtol=TOL, atol=floor)
    _assert_healthy()
