"""The ConvBlock convolution of the stage-kernel chain on tcgen05 (precision "tf32", csrc/mmx_conv_tc5.cuh) against an fp64
reference: the C ABI kernel by kernel (mmx_conv2d_large_{fwd,wgrad}_prec, forward, data gradient, weight gradient), and the
ConvMixer with set_precision("tf32") against the oracle at the model bar.

Kernel bar: 2e-4 relative per tensor (max|got-want| <= 2e-4 max|want|), as for the other tcgen05 kernels
(tests/test_gpu_io_tc5.py): bf16 hi+lo operands leave about 2^-16 per product; a product that drops a cross term is off by
about 2e-3.  Every served case also checks that the tcgen05 kernel ran (mmx_conv2d_tc5_serves, and the tf32 result differs
from the fp32 one), a NaN canary past every output, accumulation onto nonzero dw / db, a sparse d(out) (~64 sequences: dw
equals those sequences' gradient, d(in) is exactly 0 elsewhere) and an unmoved mmx_tc5_abort_count().  Shapes the kernels
decline give the fp32 result."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import mixer_np as O
from tests import masks_np as MK
from tests.golden_util import Golden, check_close, grad_scale
from tests.synthetic import synthetic_pose_windows

BAR = 2e-4
MODEL_BAR = 2e-3
ATOMIC_ORDER = 1e-5     # fp32 weight gradients summed by atomics from several CTAs: the order varies
FP32, TF32 = 0, 1
N_SPARSE = 64


# ------------------------------------------------------------------------------------------ fp64 reference
def _pad(x, kt, kp, pt, pp):
    return np.pad(x, ((0, 0), (0, 0), (pt, kt - 1 - pt), (pp, kp - 1 - pp)))


def conv_ref(x, w, b, pt, pp):
    """out[b,co,t,e] = bias[co] + sum w[co,ci,i,j] x[b,ci,t+i-pt,e+j-pp] (zero outside)."""
    Bn, Cn, T, E = x.shape
    kt, kp = w.shape[2:]
    xp = _pad(x, kt, kp, pt, pp)
    out = np.zeros((Bn, Cn, T, E)) + (0.0 if b is None else b[None, :, None, None])
    for i in range(kt):
        for j in range(kp):
            out += np.einsum("oc,bcte->bote", w[:, :, i, j], xp[:, :, i:i + T, j:j + E])
    return out


def conv_bwd_ref(x, w, dz, pt, pp):
    """d(in), dw, db of the same."""
    Bn, Cn, T, E = x.shape
    kt, kp = w.shape[2:]
    xp = _pad(x, kt, kp, pt, pp)
    dxp = np.zeros_like(xp)
    dw = np.zeros_like(w)
    for i in range(kt):
        for j in range(kp):
            dxp[:, :, i:i + T, j:j + E] += np.einsum("oc,bote->bcte", w[:, :, i, j], dz)
            dw[:, :, i, j] = np.einsum("bote,bcte->oc", dz, xp[:, :, i:i + T, j:j + E])
    return dxp[:, :, pt:pt + T, pp:pp + E], dw, dz.sum((0, 2, 3))


def test_reference_matches_float64_conv2d():
    """The reference above against torch.nn.functional.conv2d and its autograd in float64 (CPU), odd and even kernels."""
    rng = np.random.default_rng(0)
    for Cn, kt, kp, pt, pp, T, E in [(3, 5, 9, 2, 4, 6, 20), (2, 2, 4, 0, 1, 5, 11), (1, 10, 5, 4, 2, 10, 9), (4, 1, 1, 0, 0, 3, 7)]:
        x, dz = rng.standard_normal((2, Cn, T, E)), rng.standard_normal((2, Cn, T, E))
        w, b = rng.standard_normal((Cn, Cn, kt, kp)), rng.standard_normal(Cn)
        xt, wt, bt = (torch.from_numpy(a).requires_grad_(True) for a in (x, w, b))
        y = torch.nn.functional.conv2d(torch.nn.functional.pad(xt, (pp, kp - 1 - pp, pt, kt - 1 - pt)), wt, bt)
        y.backward(torch.from_numpy(dz))
        np.testing.assert_allclose(conv_ref(x, w, b, pt, pp), y.detach().numpy(), rtol=1e-12, atol=1e-11)
        for got, want in zip(conv_bwd_ref(x, w, dz, pt, pp), (xt.grad, wt.grad, bt.grad)):
            np.testing.assert_allclose(got, want.numpy(), rtol=1e-12, atol=1e-10)


# ------------------------------------------------------------------------------------------ C ABI
def _lib():
    from motionmixerconv_b200 import _lib as L
    return L.load()


def _desc(B, Cn, T, E, kt, kp, pt, pp):
    from motionmixerconv_b200 import functional as F_
    return F_.conv_half_desc(B, Cn, T, E, (kt, kp), (pt, pp), 0, "gelu", False, False, False, 0, 0.0, 0, 0)


def _p(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def _canaried(n, offset=0):
    """A device buffer of n floats followed by a NaN tail of 4096 floats; ``offset`` floats of misalignment in front."""
    buf = torch.full((offset + n + 4096,), float("nan"), device="cuda")
    return buf, buf[offset:offset + n]


def _check(name, got, want, bar=BAR):
    err = float(np.abs(got - want).max())
    scale = float(np.abs(want).max())
    assert err <= bar * scale, "%s: max err %.3g > %.1g x %.3g" % (name, err, bar, scale)


def _sparse(B, seed):
    if B <= N_SPARSE:
        return np.arange(B)
    rng = np.random.default_rng(seed)
    return np.unique(np.concatenate([[0, B - 1], rng.choice(np.arange(1, B - 1), N_SPARSE - 2, replace=False)]))


def _run_abi(lib, d, prec, xin, w, b, dz, n, dw0, db0, offset=0):
    """fwd, data gradient, wgrad through the _prec entry points.  Returns (out, d(in), dw - dw0, db - db0) and the canaries."""
    numel = xin.numel()
    ob, out = _canaried(numel, offset)
    gb, dn = _canaried(numel, offset)
    wb, dw = _canaried(dw0.numel(), offset)
    bb, db = _canaried(db0.numel(), offset)
    dw.copy_(dw0.flatten())
    db.copy_(db0)
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    assert lib.mmx_conv2d_large_fwd_prec(C.byref(d), 0, _p(xin), _p(w), _p(b), _p(out), prec, st) == 0, lib.mmx_last_error()
    assert lib.mmx_conv2d_large_fwd_prec(C.byref(d), 1, _p(dz), _p(w), None, _p(dn), prec, st) == 0, lib.mmx_last_error()
    assert lib.mmx_conv2d_large_wgrad_prec(C.byref(d), _p(dz), _p(n), _p(dw), _p(db), prec, st) == 0, lib.mmx_last_error()
    torch.cuda.synchronize()
    for nm, buf, k in (("out", ob, numel), ("d(in)", gb, numel), ("dw", wb, dw0.numel()), ("db", bb, db0.numel())):
        assert torch.isnan(buf[offset + k:]).all(), "%s: written past the end" % nm
    sh = tuple(xin.shape)
    f64 = lambda t: t.cpu().double().numpy()
    return (f64(out).reshape(sh), f64(dn).reshape(sh), f64(dw).reshape(dw0.shape) - f64(dw0), f64(db) - f64(db0))


def _data(B, Cn, T, E, kt, kp, seed):
    rng = np.random.default_rng(seed)
    x = rng.standard_normal((B, Cn, T, E)).astype(np.float32)
    n = (0.5 + rng.standard_normal((B, Cn, T, E))).astype(np.float32)
    w = (rng.standard_normal((Cn, Cn, kt, kp)) / np.sqrt(Cn * kt * kp)).astype(np.float32)
    b = (0.3 * rng.standard_normal(Cn)).astype(np.float32)
    q = _sparse(B, seed)
    dz = np.zeros((B, Cn, T, E), np.float32)
    dz[q] = rng.standard_normal((len(q), Cn, T, E)).astype(np.float32)
    dw0 = rng.standard_normal((Cn, Cn, kt, kp)).astype(np.float32)
    db0 = rng.standard_normal(Cn).astype(np.float32)
    return x, n, w, b, dz, dw0, db0, q


# (C, kt, kp, pt, pp, T, E, B): odd and even kernels (asymmetric 'same' padding), the (10, k) second convolutions, E not a
# multiple of the window, T = 6 / 10; B = 3 (one ragged item per window), and batches with >= 3 items per CTA, ragged last window
SERVED = [
    (1, 1, 1, 0, 0, 10, 40, 3), (2, 1, 3, 0, 1, 6, 64, 5), (3, 5, 5, 2, 2, 10, 50, 3), (4, 5, 9, 2, 4, 10, 192, 3),
    (8, 9, 5, 4, 2, 10, 64, 2), (8, 9, 9, 4, 4, 10, 192, 2), (8, 9, 29, 4, 14, 10, 192, 3), (8, 10, 5, 4, 2, 10, 192, 2),
    (3, 2, 4, 0, 1, 6, 40, 4), (2, 1, 28, 0, 13, 10, 64, 3), (8, 5, 9, 2, 4, 6, 192, 2), (1, 9, 29, 4, 14, 10, 40, 2),
    (8, 9, 29, 4, 14, 10, 150, 260), (4, 5, 9, 2, 4, 10, 190, 600), (8, 5, 5, 2, 2, 6, 64, 700),
]


@pytest.mark.gpu
@pytest.mark.parametrize("case", SERVED, ids=lambda c: "c%d_k%dx%d_p%d%d_t%d_e%d_b%d" % c)
def test_conv_tc5_vs_fp64(case):
    Cn, kt, kp, pt, pp, T, E, B = case
    lib = _lib()
    d = _desc(B, Cn, T, E, kt, kp, pt, pp)
    assert lib.mmx_conv2d_tc5_serves(C.byref(d)) == 1
    x, n, w, b, dz, dw0, db0, q = _data(B, Cn, T, E, kt, kp, seed=B * 31 + kp)
    dev = [torch.from_numpy(a).cuda() for a in (x, w, b, dz, n, dw0, db0)]
    aborts = lib.mmx_tc5_abort_count()
    got = _run_abi(lib, d, TF32, *dev)
    assert lib.mmx_tc5_abort_count() == aborts
    ref32 = _run_abi(lib, d, FP32, *dev)
    x64, n64, w64, dz64 = (a.astype(np.float64) for a in (x[q], n[q], w, dz[q]))
    want_out = conv_ref(x64, w64, b.astype(np.float64), pt, pp)
    want_dn, want_dw, want_db = conv_bwd_ref(n64, w64, dz64, pt, pp)
    _check("out", got[0][q], want_out)
    _check("d(in)", got[1][q], want_dn)
    _check("dw", got[2], want_dw)
    _check("db", got[3], want_db)
    rest = np.setdiff1d(np.arange(B), q)
    assert not np.any(got[1][rest]), "d(in) nonzero outside the sequences with a nonzero d(out)"
    for nm, a, r in zip(("out", "d(in)", "dw"), got[:3], ref32[:3]):
        assert not np.array_equal(a, r), "%s: tf32 equals fp32 -- the tcgen05 kernel did not run" % nm


def test_sparse_batch_construction_is_exact():
    """CPU: the weight gradient of a batch whose d(out) is zero outside q equals that of the q sequences alone, d(in) is 0 elsewhere."""
    x, n, w, b, dz, dw0, db0, q = _data(70, 2, 4, 9, 3, 5, seed=1)
    full = conv_bwd_ref(n.astype(np.float64), w.astype(np.float64), dz.astype(np.float64), 1, 2)
    part = conv_bwd_ref(n[q].astype(np.float64), w.astype(np.float64), dz[q].astype(np.float64), 1, 2)
    np.testing.assert_allclose(full[1], part[1], rtol=1e-12, atol=1e-12)
    np.testing.assert_allclose(full[2], part[2], rtol=1e-12, atol=1e-12)
    assert not np.any(full[0][np.setdiff1d(np.arange(70), q)])


@pytest.mark.gpu
def test_misaligned_pointers_are_served():
    """Plain loads and stores: tensors offset by one float still run on tcgen05, and match the reference."""
    Cn, kt, kp, pt, pp, T, E, B = 8, 5, 9, 2, 4, 10, 64, 3
    lib = _lib()
    d = _desc(B, Cn, T, E, kt, kp, pt, pp)
    x, n, w, b, dz, dw0, db0, q = _data(B, Cn, T, E, kt, kp, seed=7)
    dev = []
    for a in (x, w, b, dz, n):
        buf = torch.empty(a.size + 1, device="cuda")
        buf[1:].copy_(torch.from_numpy(a.ravel()))
        dev.append(buf[1:].view(a.shape))
    got = _run_abi(lib, d, TF32, *dev, torch.from_numpy(dw0).cuda(), torch.from_numpy(db0).cuda(), offset=1)
    ref32 = _run_abi(lib, d, FP32, *dev, torch.from_numpy(dw0).cuda(), torch.from_numpy(db0).cuda(), offset=1)
    x64, n64, w64, dz64 = (a.astype(np.float64) for a in (x, n, w, dz))
    _check("out", got[0], conv_ref(x64, w64, b.astype(np.float64), pt, pp))
    for nm, g, want in zip(("d(in)", "dw", "db"), got[1:], conv_bwd_ref(n64, w64, dz64, pt, pp)):
        _check(nm, g, want)
    assert not np.array_equal(got[0], ref32[0])


# shapes the tcgen05 kernels decline: C * round_up(kp, 8) > 256, kt * C > 128, a slab beyond shared memory (T = 40)
UNSERVED = [(8, 3, 33, 1, 16, 10, 64, 3), (8, 17, 3, 8, 1, 20, 40, 2), (8, 9, 9, 4, 4, 40, 192, 2)]


@pytest.mark.gpu
@pytest.mark.parametrize("case", UNSERVED, ids=lambda c: "c%d_k%dx%d_t%d_e%d" % (c[0], c[1], c[2], c[5], c[6]))
def test_unserved_shapes_give_the_fp32_result(case):
    Cn, kt, kp, pt, pp, T, E, B = case
    lib = _lib()
    d = _desc(B, Cn, T, E, kt, kp, pt, pp)
    assert lib.mmx_conv2d_tc5_serves(C.byref(d)) == 0
    x, n, w, b, dz, dw0, db0, q = _data(B, Cn, T, E, kt, kp, seed=3)
    dev = [torch.from_numpy(a).cuda() for a in (x, w, b, dz, n, dw0, db0)]
    got, ref = _run_abi(lib, d, TF32, *dev), _run_abi(lib, d, FP32, *dev)
    assert np.array_equal(got[0], ref[0]) and np.array_equal(got[1], ref[1])
    for g, r in zip(got[2:], ref[2:]):
        assert float(np.abs(g - r).max()) <= ATOMIC_ORDER * float(np.abs(r).max())


# ------------------------------------------------------------------------------------------ the model in precision "tf32"
def _build(cfg, params):
    from motionmixerconv_b200.conv_mixer_model import ConvMixer
    torch.manual_seed(3)
    m = ConvMixer(**cfg)
    m.load_state_dict({k: torch.from_numpy(np.asarray(v)) for k, v in params.items()}, strict=True)
    return m.cuda()


def _run(model, x, gt):
    from motionmixerconv_b200.functional import mpjpe_error
    model.zero_grad()
    xg = torch.from_numpy(x).cuda().requires_grad_(True)
    pred = model(xg)
    loss = mpjpe_error(pred, torch.from_numpy(gt).cuda())
    loss.backward()
    torch.cuda.synchronize()
    grads = {k: p.grad.detach().cpu().numpy() for k, p in model.named_parameters()}
    return pred.detach().cpu().numpy(), float(loss.detach()), grads, xg.grad.cpu().numpy()


def _halves(model):
    return [(mb, h) for mb in model.Mixer_Block for h in ((0, 1) if mb.mode_conv == "twice" else (0,))]


def _compare_oracle(got, cfg, params, x, gt, masks=None):
    pred, loss, grads, dx = got
    o64 = O.ConvMixerOracle(cfg, params, dtype=np.float64)
    p64 = o64.forward(x, training=True, masks=masks)
    l64, dp64 = O.mpjpe(p64, gt.astype(np.float64))
    g64, dx64 = o64.backward(dp64)
    check_close("pred", pred, p64.astype(np.float32), p64, rtol=MODEL_BAR)
    assert abs(loss - l64) <= MODEL_BAR * abs(l64)
    floor = 5e-6 * grad_scale(g64)
    for k in O.trainable_keys(params):
        if ".se2." in k:
            continue
        check_close("grad " + k, grads[k], g64[k].astype(np.float32), g64[k], rtol=MODEL_BAR,
                    atol=floor * (50 if k == "encoder.channelUpscaling.bias" else 1))
    check_close("dx", dx, dx64.astype(np.float32), dx64, rtol=MODEL_BAR, atol=1e-6 * float(np.abs(dx64).max()))


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["conv_c8_k5x9", "conv_k3", "conv_k3_bn", "conv_maxpool_bn", "conv_evenk"])
def test_golden_fixtures_in_tf32(case, monkeypatch):
    """The fixtures generated from the reference in precision "tf32", every half on the stage-kernel chain (forced where the
    fused kernels serve it), against the fp64 oracle at the model bar; each of those halves runs its convolution on tcgen05."""
    g = Golden(case)
    model = _build(g.cfg, g.params).set_precision("tf32")
    model.train()
    B = len(g.x)
    if not all(mb.uses_large_path(h, B) for mb, h in _halves(model)):
        monkeypatch.setenv("MMX_CONV_FORCE_LARGE", "1")
    assert all(mb.uses_large_path(h, B) and mb.uses_tc5_conv(h, B) for mb, h in _halves(model))
    lib = _lib()
    aborts = lib.mmx_tc5_abort_count()
    got = _run(model, g.x, g.gt)
    assert lib.mmx_tc5_abort_count() == aborts
    _compare_oracle(got, g.cfg, g.params, g.x, g.gt)
    fp = _run(_build(g.cfg, g.params).train(), g.x, g.gt)
    assert not np.array_equal(got[0], fp[0]), "tf32 equals fp32: the tcgen05 convolution did not run"


BASE = dict(num_blocks=2, dimPosIn=33, dimPosEmb=192, dimPosOut=33, in_nTP=10, out_nTP=10, conv_nChan=8, activation="mish",
            use_se=True, r_se=8, encoder_n_harmonic_functions=0, encoder_omega0=0)


def _fresh(cfg, seed=3):
    from motionmixerconv_b200.conv_mixer_model import ConvMixer
    torch.manual_seed(seed)
    m = ConvMixer(**cfg)
    return m, {k: v.detach().cpu().numpy().copy() for k, v in m.state_dict().items()}


@pytest.mark.gpu
def test_dropout_in_tf32_vs_oracle_with_the_same_masks():
    cfg = dict(BASE, conv1_kernel_shape=(5, 9), mode_conv="twice", regularization=0.1, num_blocks=1)
    m, params = _fresh(cfg, seed=4321)
    model = m.cuda().set_precision("tf32").train()
    assert all(mb.uses_tc5_conv(h, 4) and mb.uses_large_path(h, 4) for mb, h in _halves(model))
    x, gt = synthetic_pose_windows(4, 10, 10, 33, scale="ais", seed=5)
    masks = MK.conv_masks(cfg, len(x), 4321, step=0)
    _compare_oracle(_run(model, x, gt), cfg, params, x, gt, masks)


@pytest.mark.gpu
def test_trainstep_in_tf32_vs_oracle_and_graph_vs_eager():
    """Three TrainStep Adam steps in tf32 against the oracle; the captured graph against eager (dw is summed over CTAs by atomics,
    so within 1e-5 rather than bit for bit)."""
    from motionmixerconv_b200.train import TrainStep
    cfg = dict(BASE, conv1_kernel_shape=(9, 29), mode_conv="once", regularization=-1.0)
    B = 6
    x, gt = synthetic_pose_windows(B, 10, 10, 33, scale="ais", seed=11)
    xs, gts = torch.from_numpy(x).cuda(), torch.from_numpy(gt).cuda()
    out = {}
    for use_graph in (False, True):
        m, params = _fresh(cfg)
        model = m.cuda().set_precision("tf32").train()
        assert all(mb.uses_tc5_conv(h, B) for mb, h in _halves(model))
        ts = TrainStep(model, lr=1e-3, weight_decay=1e-5, use_cuda_graph=use_graph)
        out[use_graph] = ([float(ts.step(xs, gts)) for _ in range(3)], {k: v.detach().cpu().numpy() for k, v in model.state_dict().items()})
    want = O.train_steps(O.ConvMixerOracle(cfg, params), x, gt, 3)
    np.testing.assert_allclose(out[False][0], want, rtol=MODEL_BAR)
    np.testing.assert_allclose(out[True][0], out[False][0], rtol=1e-5)
    for k, v in out[False][1].items():
        if v.dtype.kind == "f":
            np.testing.assert_allclose(out[True][1][k], v, rtol=1e-5, atol=1e-5 * max(1.0, float(np.abs(v).max())), err_msg=k)


@pytest.mark.gpu
def test_optuna_cell_at_many_tiles_per_cta_replicated_batch(monkeypatch):
    """The Optuna 5x5 cell (C = 8, E = 192; two windows per sequence) on the chain at B = 1031: 2062 work items, >= 8 x SMs.
    Every prediction row and dx row against the oracle of the base sequences."""
    from tests.test_gpu_large_batch import P, replicated_oracle
    monkeypatch.setenv("MMX_CONV_FORCE_LARGE", "1")
    cfg = dict(BASE, conv1_kernel_shape=(5, 5), mode_conv="once", regularization=0, num_blocks=1)
    m, params = _fresh(cfg)
    model = m.cuda().set_precision("tf32").train()
    B = P
    assert all(mb.uses_tc5_conv(h, B) and mb.uses_large_path(h, B) for mb, h in _halves(model))
    xb, gtb = synthetic_pose_windows(P, 10, 10, 33, scale="ais", seed=21)
    idx = np.arange(B) % P
    pred, loss, grads, dx = _run(model, xb[idx], gtb[idx])
    rep = replicated_oracle(O.ConvMixerOracle(cfg, params, dtype=np.float64), xb, gtb, B)
    check_close("pred", pred, rep.pred[idx].astype(np.float32), rep.pred[idx], rtol=MODEL_BAR)
    check_close("dx", dx, rep.dx[idx].astype(np.float32), rep.dx[idx], rtol=MODEL_BAR, atol=1e-6 * float(np.abs(rep.dx).max()))
    floor = 5e-6 * grad_scale(rep.grads)
    for k in O.trainable_keys(params):
        if ".se2." in k:
            continue
        check_close("grad " + k, grads[k], rep.grads[k].astype(np.float32), rep.grads[k], rtol=MODEL_BAR,
                    atol=floor * (50 if k == "encoder.channelUpscaling.bias" else 1))


# ------------------------------------------------------------------------------------------ opt-in
def test_precision_is_not_a_constructor_argument_nor_state():
    import inspect
    from motionmixerconv_b200.conv_mixer_model import ConvMixer
    assert "precision" not in inspect.signature(ConvMixer.__init__).parameters
    m, sd = _fresh(dict(BASE, conv1_kernel_shape=(5, 9), regularization=0))
    assert m.set_precision("tf32") is m
    assert list(m.state_dict()) == list(sd)
    with pytest.raises(ValueError):
        m.set_precision("bf16")


@pytest.mark.gpu
def test_default_convmixer_stays_fp32_under_mmx_precision_tf32(monkeypatch):
    """MMX_PRECISION=tf32 / functional.set_precision("tf32") leave a default ConvMixer in fp32, bit for bit."""
    from motionmixerconv_b200 import functional as F_
    cfg = dict(BASE, conv1_kernel_shape=(5, 9), mode_conv="twice", regularization=0, num_blocks=1)
    x, gt = synthetic_pose_windows(3, 10, 10, 33, scale="ais", seed=2)
    base = _run(_fresh(cfg)[0].cuda().train(), x, gt)
    old = F_.get_precision()
    monkeypatch.setenv("MMX_PRECISION", "tf32")
    try:
        F_.set_precision("tf32")
        got = _run(_fresh(cfg)[0].cuda().train(), x, gt)
    finally:
        F_.set_precision(old)
    for a, b in zip((got[0], got[3]), (base[0], base[3])):
        assert np.array_equal(a, b)
