"""GPU (-m gpu): the tcgen05 / TMEM MixerBlock kernel family (precision="tf32": channel half on the tensor cores with
bf16x3 split operands, token half on packed-fp32 CUDA cores; csrc/mmx_chan_tc5.cuh, csrc/mmx_tok.cuh) through the product
modules / C ABI against the golden fixtures (generated from the reference) and the numpy oracle.

Tolerance: the north star's reduced-precision bar, 2e-3 relative per tensor, for EVERY tensor (predictions, loss, input
gradient, all parameter gradients, any batch size) -- no loosened cases.  Measured: 5e-6 ... 3e-5.
"""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import mixer_np as O
from tests import masks_np as MK
from tests.golden_util import Golden, check_close, grad_scale
from tests.synthetic import synthetic_pose_windows

pytestmark = pytest.mark.gpu
TOL = 2e-3


def _model(cfg, params=None, seed=0):
    from motionmixerconv_b200.mlp_mixer import MlpMixer
    torch.manual_seed(seed)
    m = MlpMixer(**cfg)
    if params is not None:
        m.load_state_dict({k: torch.from_numpy(np.asarray(v)) for k, v in params.items()}, strict=True)
    return m.cuda().set_precision("tf32")


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


def _oracle(cfg, params, x, gt, masks=None):
    o = O.MlpMixerOracle(cfg, params, dtype=np.float64)
    p = o.forward(x, training=True, masks=masks)
    l, dp = O.mpjpe(p, gt.astype(np.float64))
    g, dx = o.backward(dp)
    return p, float(l), g, dx


def _compare(pred, loss, grads, dx, want, tol=TOL):
    p64, l64, g64, dx64 = want
    check_close("pred", pred, p64, rtol=tol)
    assert abs(loss - l64) <= tol * abs(l64)
    floor = 0.01 * tol * grad_scale(g64)          # tensors two orders below the gradient scale are cancellation noise
    for k, w in g64.items():
        if k in grads:
            check_close("grad " + k, grads[k], w, rtol=tol, atol=floor)
    check_close("dx", dx, dx64, rtol=tol)


def _assert_healthy():
    from motionmixerconv_b200 import _lib as L
    assert L.load().mmx_tc5_abort_count() == 0            # no pipeline wait ever timed out


def test_the_tcgen05_family_is_what_runs():
    """precision="tf32" must change the arithmetic (else these tests would silently exercise the FP32 kernels), and the
    descriptor must be one the family serves (mmx_mlp_block_saves is its capability bit)."""
    from motionmixerconv_b200 import _lib as L
    from motionmixerconv_b200 import functional as F_
    g = Golden("mlp_k2")
    m = _model(g.cfg, g.params).eval()
    x = torch.from_numpy(g.x).cuda()
    with torch.no_grad():
        a = m(x)
        b = m.set_precision("fp32")(x)
    d = (a - b).abs().max().item() / b.abs().max().item()
    assert 0.0 < d < TOL, d
    desc = F_.mlp_block_desc(64, 10, 50, 20, 50, 1, "mish", True, False, True, 0, 0.0, 0, 0, "tf32")
    assert L.load().mmx_mlp_block_saves(C.byref(desc)) == 1
    desc = F_.mlp_block_desc(64, 10, 50, 20, 50, 1, "mish", True, False, True, 0, 0.0, 0, 0, "fp32")
    assert L.load().mmx_mlp_block_saves(C.byref(desc)) == 0
    _assert_healthy()


def test_golden_k2():
    g = Golden("mlp_k2")
    cfg = dict(g.cfg)
    model = _model(cfg, g.params).train()
    pred, loss, grads, dx = _run(model, g.x, g.gt)
    check_close("pred vs reference", pred, g.pred, rtol=TOL)
    assert abs(loss - g.loss) <= TOL * abs(g.loss)
    floor = 0.01 * TOL * grad_scale(g.grads)
    for k, want in g.grads.items():
        check_close("grad " + k, grads[k], want, rtol=TOL, atol=floor)      # 6 sequences
    check_close("dx", dx, g.dx, rtol=TOL)
    model.eval()
    with torch.no_grad():
        pe = model(torch.from_numpy(g.x).cuda()).cpu().numpy()
    check_close("pred_eval", pe, g.pred_eval, rtol=TOL)
    _assert_healthy()


@pytest.mark.parametrize("B", [1, 2, 11, 12, 13, 333, 1000, 4096, 4097])
def test_ragged_batches_vs_oracle(B):
    """Batch sizes around the 12-sequence MMA tile / 5-sequence token tile: partial tiles, a single sequence, several tiles
    per CTA (B = 4096 is the benchmark size: 342 MMA tiles on 148 CTAs)."""
    g = Golden("mlp_k2")
    c = dict(g.cfg, regularization=0)
    x, gt = synthetic_pose_windows(B, c["seq_len"], c["pred_len"], c["input_size"], scale="amass", seed=7)
    model = _model(c, g.params).train()
    _compare(*_run(model, x, gt), _oracle(c, g.params, x, gt))
    _assert_healthy()


VARIANTS = {
    "gelu_h32_ch40": dict(hidden_dim=32, channels_mlp_dim=40, activation="gelu"),
    "no_se": dict(use_se=False),
    "se_hidden_2": dict(r_se=4),
    "h48_ch24": dict(hidden_dim=48, channels_mlp_dim=24),
    "h64_ch64_gelu": dict(hidden_dim=64, channels_mlp_dim=64, activation="gelu"),      # streamed weights at operand width 64
    "h78_ch30": dict(hidden_dim=78, channels_mlp_dim=30),
    "h72_ch72": dict(hidden_dim=72, channels_mlp_dim=72),                              # resident KP = 80, 4-float row loads
    "h50_ch49": dict(hidden_dim=50, channels_mlp_dim=49),                              # odd ch: resident KP = 64 only
    "h64_ch63": dict(hidden_dim=64, channels_mlp_dim=63),                              # odd ch: resident KP = 80 only
    "tok7_T8": dict(tokens_mlp_dim=7, seq_len=8, pred_len=8),                          # generic-T instantiation (T != 10)
    "T16_to25": dict(seq_len=16, pred_len=25, tokens_mlp_dim=32, r_se=8),              # two sequences per warp, SE hidden 2
    "T13_h52": dict(seq_len=13, hidden_dim=52, channels_mlp_dim=52, r_se=4),           # two sequences per warp, 6 idle lanes
    "T6_h40": dict(seq_len=6, hidden_dim=40, channels_mlp_dim=40, r_se=2),             # five sequences per warp, SE hidden 3
}


@pytest.mark.parametrize("name", sorted(VARIANTS))
def test_shape_variants_vs_oracle(name):
    from motionmixerconv_b200 import _lib as L
    from motionmixerconv_b200 import functional as F_
    cfg = dict(Golden("mlp_k2").cfg, num_blocks=2, regularization=0, **VARIANTS[name])
    model = _model(cfg, None, seed=3).train()
    mb = model.Mixer_Block[0]
    desc = F_.mlp_block_desc(515, mb.seq_len, mb.hidden_dim, *mb.meta())
    assert L.load().mmx_mlp_block_saves(C.byref(desc)) == 1         # the tcgen05 family serves it (no FP32 fall-back)
    params = {k: v.detach().cpu().numpy() for k, v in model.state_dict().items()}
    x, gt = synthetic_pose_windows(515, cfg["seq_len"], cfg["pred_len"], 66, scale="amass", seed=9)
    _compare(*_run(model, x, gt), _oracle(cfg, params, x, gt))
    _assert_healthy()


def test_save_variant_equals_recompute_variant():
    """mmx_mlp_block_fwd_save / _bwd_saved (x1 + gates handed to the backward) against mmx_mlp_block_fwd / _bwd (everything
    recomputed from x): same outputs bit for bit, gradients within rounding of each other."""
    from motionmixerconv_b200 import _lib as L
    from motionmixerconv_b200 import functional as F_
    torch.manual_seed(0)
    B, T, H, tok, ch = 1000, 10, 50, 20, 50
    lib = L.load()
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    shapes = [(H,), (H,), (tok, T), (tok,), (T, tok), (T,), (H,), (H,), (ch, H), (ch,), (H, ch), (H,), (1, T), (T, 1)]
    params = [torch.randn(*s, device="cuda") * 0.3 for s in shapes]
    params[0] += 1.0
    params[6] += 1.0
    x, dy = torch.randn(B, T, H, device="cuda"), torch.randn(B, T, H, device="cuda")
    desc = F_.mlp_block_desc(B, T, H, tok, ch, 1, "mish", True, False, True, 1, 0.1, 1234, 5, "tf32")
    tw = F_.mlp_block_table(params)

    def run(saved):
        y, dx = torch.empty_like(x), torch.empty_like(x)
        grads = [torch.zeros_like(p) for p in params]
        tg = F_.mlp_block_table(grads)
        if saved:
            x1, gate = torch.empty_like(x), torch.empty(B, T, device="cuda")
            L.check(lib, lib.mmx_mlp_block_fwd_save(C.byref(desc), C.byref(tw), x.data_ptr(), y.data_ptr(), x1.data_ptr(), gate.data_ptr(), st), "fwd")
            L.check(lib, lib.mmx_mlp_block_bwd_saved(C.byref(desc), C.byref(tw), C.byref(tg), x.data_ptr(), x1.data_ptr(), gate.data_ptr(),
                                                     dy.data_ptr(), dx.data_ptr(), st), "bwd")
        else:
            L.check(lib, lib.mmx_mlp_block_fwd(C.byref(desc), C.byref(tw), x.data_ptr(), y.data_ptr(), st), "fwd")
            L.check(lib, lib.mmx_mlp_block_bwd(C.byref(desc), C.byref(tw), C.byref(tg), x.data_ptr(), dy.data_ptr(), dx.data_ptr(), st), "bwd")
        torch.cuda.synchronize()
        return y, dx, grads

    ya, dxa, ga = run(False)
    yb, dxb, gb = run(True)
    assert torch.equal(ya, yb)
    assert (dxa - dxb).abs().max().item() <= 1e-4 * dxa.abs().max().item()
    for a, b in zip(ga, gb):
        assert (a - b).abs().max().item() <= 1e-4 * max(a.abs().max().item(), 1e-6)
    _assert_healthy()


def test_dropout_mask_generator_matches_its_numpy_twin():
    """Pins tests/masks_np.tc5_mask (the masks the oracle gets in the tests below) to the device generator, bit for bit."""
    from motionmixerconv_b200 import _lib as L
    lib = L.load()
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    for rows, W, p, seed, site, step in [(37, 50, 0.1, 1234, 2, 0), (500, 30, 0.25, (7 << 40) + 99, 12, 3), (64, 64, 0.5, 1, 7, 100000)]:
        out = torch.empty(rows, W, device="cuda")
        d = L.MmxDropout(p, seed, step, None)
        L.check(lib, lib.mmx_tc5_dropout_mask(C.byref(d), site, rows, W, out.data_ptr(), st), "mask")
        torch.cuda.synchronize()
        want = MK.tc5_mask(rows, W, p, seed, site, step)
        assert np.array_equal(out.cpu().numpy(), want)
        assert abs(float((want == 0).mean()) - p) < 0.05


@pytest.mark.parametrize("B", [6, 333])
def test_dropout_forward_and_backward_vs_oracle_with_the_same_masks(B):
    """The benchmarked configuration (dropout 0.1): the oracle is given the masks the kernels draw (numpy twin of the
    generator) and every tensor is compared -- not just 'masks differ, gradients finite'."""
    g = Golden("mlp_k2")
    c = dict(g.cfg, regularization=0.1)
    x, gt = (g.x, g.gt) if B == 6 else synthetic_pose_windows(B, 10, 10, 66, scale="h36m", seed=21)
    torch.manual_seed(4321)
    model = _model(c, g.params, seed=4321).train()
    masks = MK.mlp_tc5_masks(c, len(x), 4321, step=0)
    got = _run(model, x, gt)
    _compare(*got, _oracle(c, g.params, x, gt, masks=masks))
    masks1 = MK.mlp_tc5_masks(c, len(x), 4321, step=1)          # second call of the modules: step 1, fresh masks
    got1 = _run(model, x, gt)
    _compare(*got1, _oracle(c, g.params, x, gt, masks=masks1))
    assert not np.array_equal(got[0], got1[0])
    _assert_healthy()


def test_unsupported_shapes_fall_back_to_fp32_kernels():
    """tf32 is a permission: H = 256 is not served by the tcgen05 family and must give the FP32 result."""
    cfg = dict(Golden("mlp_k2").cfg, num_blocks=1, hidden_dim=256, channels_mlp_dim=64)
    m = _model(cfg, None, seed=1).eval()
    x = torch.from_numpy(synthetic_pose_windows(9, 10, 10, 66, scale="amass", seed=2)[0]).cuda()
    with torch.no_grad():
        a = m(x)
        b = m.set_precision("fp32")(x)
    assert torch.equal(a, b)


# ------------------------------------------------------------------------------------------ wide variant (80 <= max(H, ch) <= 128)
def test_wide_family_serves_k4():
    """K4 (AMASS-shaped, H = ch = 128): the wide tcgen05 channel half (csrc/mmx_chan_wide.cuh) is what runs."""
    from motionmixerconv_b200 import _lib as L
    from motionmixerconv_b200 import functional as F_
    for H, ch, want in [(128, 128, 1), (96, 128, 1), (128, 80, 1), (130, 64, 0), (64, 130, 0), (128, 127, 0)]:
        desc = F_.mlp_block_desc(64, 10, H, 20, ch, 1, "gelu", True, False, True, 0, 0.0, 0, 0, "tf32")
        assert L.load().mmx_mlp_block_saves(C.byref(desc)) == want, (H, ch)
    g = Golden("mlp_k4")
    m = _model(g.cfg, g.params).eval()
    x = torch.from_numpy(g.x).cuda()
    with torch.no_grad():
        a = m(x)
        b = m.set_precision("fp32")(x)
    d = (a - b).abs().max().item() / b.abs().max().item()
    assert 0.0 < d < TOL, d
    _assert_healthy()


def test_golden_k4():
    g = Golden("mlp_k4")
    model = _model(dict(g.cfg), g.params).train()
    pred, loss, grads, dx = _run(model, g.x, g.gt)
    check_close("pred vs reference", pred, g.pred, rtol=TOL)
    assert abs(loss - g.loss) <= TOL * abs(g.loss)
    floor = 0.01 * TOL * grad_scale(g.grads)
    for k, want in g.grads.items():
        check_close("grad " + k, grads[k], want, rtol=TOL, atol=floor)
    check_close("dx", dx, g.dx, rtol=TOL)
    model.eval()
    with torch.no_grad():
        pe = model(torch.from_numpy(g.x).cuda()).cpu().numpy()
    check_close("pred_eval", pe, g.pred_eval, rtol=TOL)
    _assert_healthy()


@pytest.mark.parametrize("B", [1, 12, 13, 333, 2000, 4096])
def test_wide_ragged_batches_vs_oracle(B):
    """K4 at batch sizes around the 12-sequence MMA tile, and the benchmark size (342 tiles on 148 CTAs: the weight slot
    cycles W1' -> W2 -> W1' several times per CTA, dW accumulates in TMEM across tiles)."""
    g = Golden("mlp_k4")
    c = dict(g.cfg, regularization=0)
    x, gt = synthetic_pose_windows(B, c["seq_len"], c["pred_len"], c["input_size"], scale="amass", seed=7)
    model = _model(c, g.params).train()
    _compare(*_run(model, x, gt), _oracle(c, g.params, x, gt))
    _assert_healthy()


WIDE_VARIANTS = {
    "h96_ch128_mish": dict(hidden_dim=96, channels_mlp_dim=128, activation="mish"),
    "h128_ch100": dict(hidden_dim=128, channels_mlp_dim=100),
    "h100_ch84_no_se": dict(hidden_dim=100, channels_mlp_dim=84, use_se=False),
    "h90_ch128": dict(hidden_dim=90, channels_mlp_dim=128, activation="mish"),          # H % 4 != 0: 8-byte row accesses
    "h80_ch80": dict(hidden_dim=80, channels_mlp_dim=80),                              # the first width the 80-column plan cannot hold
    "h128_T16": dict(hidden_dim=128, channels_mlp_dim=128, seq_len=16, pred_len=25, tokens_mlp_dim=32, r_se=8),
}


@pytest.mark.parametrize("name", sorted(WIDE_VARIANTS))
def test_wide_shape_variants_vs_oracle(name):
    cfg = dict(Golden("mlp_k4").cfg, num_blocks=2, regularization=0, **WIDE_VARIANTS[name])
    model = _model(cfg, None, seed=3).train()
    params = {k: v.detach().cpu().numpy() for k, v in model.state_dict().items()}
    x, gt = synthetic_pose_windows(301, cfg["seq_len"], cfg["pred_len"], cfg["input_size"], scale="amass", seed=9)
    _compare(*_run(model, x, gt), _oracle(cfg, params, x, gt))
    _assert_healthy()


def test_wide_dropout_vs_oracle_with_the_same_masks():
    g = Golden("mlp_k4")
    c = dict(g.cfg, regularization=0.1)
    x, gt = synthetic_pose_windows(77, c["seq_len"], c["pred_len"], c["input_size"], scale="amass", seed=21)
    torch.manual_seed(4321)
    model = _model(c, g.params, seed=4321).train()
    masks = MK.mlp_tc5_masks(c, len(x), 4321, step=0)
    _compare(*_run(model, x, gt), _oracle(c, g.params, x, gt, masks=masks))
    _assert_healthy()


def test_wide_save_variant_and_in_place_recompute_variant_agree():
    from motionmixerconv_b200 import _lib as L
    from motionmixerconv_b200 import functional as F_
    torch.manual_seed(0)
    B, T, H, tok, ch = 500, 10, 128, 20, 128
    lib = L.load()
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    shapes = [(H,), (H,), (tok, T), (tok,), (T, tok), (T,), (H,), (H,), (ch, H), (ch,), (H, ch), (H,), (1, T), (T, 1)]
    params = [torch.randn(*s, device="cuda") * 0.2 for s in shapes]
    params[0] += 1.0
    params[6] += 1.0
    x, dy = torch.randn(B, T, H, device="cuda"), torch.randn(B, T, H, device="cuda")
    desc = F_.mlp_block_desc(B, T, H, tok, ch, 1, "gelu", True, False, True, 1, 0.1, 1234, 5, "tf32")
    tw = F_.mlp_block_table(params)

    def run(saved):
        y, dx = torch.empty_like(x), torch.empty_like(x)
        grads = [torch.zeros_like(p) for p in params]
        tg = F_.mlp_block_table(grads)
        if saved:
            x1, gate = torch.empty_like(x), torch.empty(B, T, device="cuda")
            L.check(lib, lib.mmx_mlp_block_fwd_save(C.byref(desc), C.byref(tw), x.data_ptr(), y.data_ptr(), x1.data_ptr(), gate.data_ptr(), st), "fwd")
            L.check(lib, lib.mmx_mlp_block_bwd_saved(C.byref(desc), C.byref(tw), C.byref(tg), x.data_ptr(), x1.data_ptr(), gate.data_ptr(),
                                                     dy.data_ptr(), dx.data_ptr(), st), "bwd")
        else:
            L.check(lib, lib.mmx_mlp_block_fwd(C.byref(desc), C.byref(tw), x.data_ptr(), y.data_ptr(), st), "fwd")
            L.check(lib, lib.mmx_mlp_block_bwd(C.byref(desc), C.byref(tw), C.byref(tg), x.data_ptr(), dy.data_ptr(), dx.data_ptr(), st), "bwd")
        torch.cuda.synchronize()
        return y, dx, grads

    ya, dxa, ga = run(False)
    yb, dxb, gb = run(True)
    assert torch.equal(ya, yb)
    assert (dxa - dxb).abs().max().item() <= 1e-4 * dxa.abs().max().item()
    for a, b in zip(ga, gb):
        assert (a - b).abs().max().item() <= 1e-4 * max(a.abs().max().item(), 1e-6)
    _assert_healthy()


def test_mpjpe_after_200_steps_within_0p1mm_of_oracle():
    """North-star criterion: MPJPE after 200 synthetic-data Adam steps within 0.1 mm of the oracle (TrainStep: CUDA graph,
    save variant of the block kernels)."""
    from motionmixerconv_b200.train import TrainStep
    g = Golden("mlp_k2")
    c = dict(g.cfg, regularization=0)
    x, gt = synthetic_pose_windows(256, 10, 10, 66, scale="h36m", seed=5)
    model = _model(c, g.params).train()
    ts = TrainStep(model, lr=1e-3, weight_decay=1e-5)
    xs, gts = torch.from_numpy(x).cuda(), torch.from_numpy(gt).cuda()
    for _ in range(200):
        loss = ts.step(xs, gts)
    want = O.train_steps(O.MlpMixerOracle(c, g.params), x, gt, 200)[-1]
    assert abs(float(loss) - want) < 0.1, (float(loss), want)           # mm
    _assert_healthy()
