"""GPU (-m gpu): ConvMixer at embedding widths up to 512.

The output head's resident tile (all of fc_out.weight plus the tile's rows) stops fitting shared memory at E = 389 (C = 1,
backward) and E = 253 (C = 8, backward); the harmonic PoseEncoder's weight chunk at E of about 200.  Past those widths the
chunked head plan and the split-harmonic encoder chunk take over (csrc/mmx_conv_io.cuh).  Checked here:
  * the PoseEncoder and head through the C ABI against the fp64 oracle (a num_blocks = 0 model is exactly encoder -> head),
    with NaN canaries past every output, gradients accumulated onto nonzero buffers and a sparse dout;
  * the chunked head forced onto a shape the resident plan serves, against the resident result;
  * whole models at E = 512 against the oracle, TrainStep with and without CUDA graphs, and the autograd path and TrainStep
    launching the same C ABI calls.
"""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import mixer_np as O
from tests import masks_np as MK
from tests.golden_util import check_close, grad_scale
from tests.synthetic import synthetic_pose_windows
from tests.test_gpu_conv_large import _build, _compare, _oracles, _run

pytestmark = pytest.mark.gpu
TOL = 1e-5
CANARY = 64


def _lib():
    from motionmixerconv_b200 import _lib as L
    return L, L.load()


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).cuda()


class Out:
    """Output buffer followed by NaN canaries; starts at g0 (accumulated gradients) or NaN."""

    def __init__(self, shape, g0=None):
        self.n = int(np.prod(shape))
        self.buf = torch.full((self.n + CANARY,), float("nan"), device="cuda")
        self.t = self.buf[:self.n].view(shape)
        self.g0 = g0
        if g0 is not None:
            self.t.copy_(torch.from_numpy(g0))

    @property
    def ptr(self):
        return self.t.data_ptr()

    def get(self, what):
        torch.cuda.synchronize()
        assert torch.isnan(self.buf[self.n:]).all(), "%s: written past its end" % what
        got = self.t.cpu().numpy()
        return got if self.g0 is None else got.astype(np.float64) - self.g0


def _cfg(C, E, Hn, D=66):
    return dict(num_blocks=0, dimPosIn=D, dimPosEmb=E, dimPosOut=66, in_nTP=10, out_nTP=25, conv_nChan=C,
                encoder_n_harmonic_functions=Hn, encoder_omega0=0.1)


def _params(cfg, seed):
    from oracle.mixer_torch import random_params
    p = {k: v.numpy().copy() for k, v in random_params("conv", cfg, seed=seed).items()}
    rng = np.random.default_rng(seed)
    E = cfg["dimPosEmb"]
    p["LN.weight"] = (1.0 + 0.3 * rng.standard_normal(E)).astype(np.float32)
    p["LN.bias"] = (0.2 * rng.standard_normal(E)).astype(np.float32)
    return p


def _abi(cfg, params, x, dout, seed):
    """encoder fwd -> head fwd -> head bwd -> encoder bwd through the C ABI; gradients accumulate onto random g0."""
    L, lib = _lib()
    B, T = x.shape[:2]
    Cn, E, To, D, Hn = cfg["conv_nChan"], cfg["dimPosEmb"], cfg["out_nTP"], cfg["dimPosOut"], cfg["encoder_n_harmonic_functions"]
    rng = np.random.default_rng(seed + 7)
    P = {k: _dev(v) for k, v in params.items() if np.asarray(v).dtype.kind == "f"}
    G = {k: Out(v.shape, g0=rng.standard_normal(v.shape).astype(np.float32)) for k, v in params.items() if k in O.trainable_keys(params)}

    def enc(src, get):
        t = L.MmxEncoderParams()
        t.freq = P["encoder.frequencies"].data_ptr() if Hn > 0 else None
        t.w, t.b = get(src, "encoder.embed_mlp.weight"), get(src, "encoder.embed_mlp.bias")
        t.wc, t.bc = get(src, "encoder.channelUpscaling.weight"), get(src, "encoder.channelUpscaling.bias")
        return t

    def head(src, get):
        t = L.MmxConvHeadParams()
        t.ln_w, t.ln_b = get(src, "LN.weight"), get(src, "LN.bias")
        t.wt, t.bt = get(src, "conv_out.weight"), get(src, "conv_out.bias")
        t.wp, t.bp = get(src, "project_channels.weight"), get(src, "project_channels.bias")
        t.wf, t.bf = get(src, "fc_out.weight"), get(src, "fc_out.bias")
        return t

    def pw(src, k):
        return src[k].data_ptr()

    def pg(src, k):
        return src[k].ptr

    xd, doutd = _dev(x), _dev(dout)
    ed, hd = L.MmxEncoderDesc(B, T, cfg["dimPosIn"], E, Cn, Hn), L.MmxConvHeadDesc(B, Cn, T, To, E, D)
    m, y, pred = Out((B * T, E)), Out((B, Cn, T, E)), Out((B, To, D))
    L.check(lib, lib.mmx_pose_encoder_fwd(C.byref(ed), C.byref(enc(P, pw)), xd.data_ptr(), m.ptr, y.ptr, _stream()), "enc fwd")
    L.check(lib, lib.mmx_conv_head_fwd(C.byref(hd), C.byref(head(P, pw)), y.ptr, pred.ptr, _stream()), "head fwd")
    dy, dm, dx = Out((B, Cn, T, E)), Out((B * T, E)), Out(x.shape)
    L.check(lib, lib.mmx_conv_head_bwd(C.byref(hd), C.byref(head(P, pw)), C.byref(head(G, pg)), y.ptr, doutd.data_ptr(), dy.ptr,
                                       _stream()), "head bwd")
    L.check(lib, lib.mmx_pose_encoder_bwd(C.byref(ed), C.byref(enc(P, pw)), C.byref(enc(G, pg)), xd.data_ptr(), m.ptr, dy.ptr,
                                          dm.ptr, dx.ptr, _stream()), "enc bwd")
    out = {"pred": pred.get("pred"), "dy": dy.get("dy"), "dx": dx.get("dx")}
    m.get("m"), y.get("y"), dm.get("dm")
    return out, {k: g.get(k) for k, g in G.items()}


def _check_abi(cfg, B, seed=3, sparse=False):
    params = _params(cfg, seed)
    x, _ = synthetic_pose_windows(B, cfg["in_nTP"], cfg["out_nTP"], cfg["dimPosIn"], scale="amass", seed=seed)
    dout = np.random.default_rng(seed + 1).standard_normal((B, cfg["out_nTP"], cfg["dimPosOut"])).astype(np.float32)
    keep = None
    if sparse:
        keep = np.zeros(B, bool)
        keep[[0, B // 2, B - 1]] = True
        dout[~keep] = 0.0
    ref = []
    for dt in (np.float32, np.float64):
        o = O.ConvMixerOracle(cfg, params, dtype=dt)
        ref.append((o.forward(x),) + o.backward(dout.astype(dt)))
    (p32, g32, dx32), (p64, g64, dx64) = ref
    got, grads = _abi(cfg, params, x, dout, seed)
    check_close("pred", got["pred"], p32, p64, rtol=TOL)
    floor = 5e-6 * grad_scale(g32)
    for k in O.trainable_keys(params):
        check_close("grad " + k, grads[k], g32[k], g64[k], rtol=TOL, atol=floor * (50 if k == "encoder.channelUpscaling.bias" else 1))
    check_close("dx", got["dx"], dx32, dx64, rtol=TOL, atol=1e-6 * float(np.abs(dx32).max()))
    if sparse:
        assert not got["dy"][~keep].any(), "dy of sequences with zero dout must be exactly 0"
        assert not got["dx"][~keep].any()
    return got


ABI = {
    # name: (C, E, Hn, B, forced chunk width, forced tile)
    "c1_e512": (1, 512, 0, 445, 0, 0),            # 445 tiles of one sequence on 148 SMs: 3 - 4 tiles per CTA
    "c8_e512": (8, 512, 0, 300, 0, 0),
    "c2_e509_harmonic16": (2, 509, 16, 37, 0, 0),  # odd E, split-harmonic encoder
    "c1_e389_first_declined": (1, 389, 0, 301, 0, 0),
    "c8_e253_first_declined": (8, 253, 4, 150, 0, 0),
    "c3_e260_ragged_tiles": (3, 260, 0, 3 * 148 * 3 + 2, 56, 3),  # >= 3 tiles per CTA, ragged last chunk and last tile
}


@pytest.mark.parametrize("case", sorted(ABI))
def test_encoder_and_head_through_the_c_abi(case, monkeypatch):
    Cn, E, Hn, B, ec, S = ABI[case]
    if ec:
        monkeypatch.setenv("MMX_CHEAD_EC", str(ec))
    if S:
        monkeypatch.setenv("MMX_CHEAD_S_FWD", str(S))
        monkeypatch.setenv("MMX_CHEAD_S_BWD", str(S))
    _check_abi(_cfg(Cn, E, Hn), B)


def test_sparse_dout_gives_exactly_zero_dy_elsewhere():
    _check_abi(_cfg(1, 512, 0), 40, sparse=True)


def test_chunked_head_forced_on_a_resident_shape(monkeypatch):
    """E = 192: the resident plan serves it; the chunked plan forced onto it agrees with it (and both with the oracle)."""
    cfg = _cfg(4, 192, 0)
    resident = _check_abi(cfg, 333)
    monkeypatch.setenv("MMX_CHEAD_EC", "40")
    chunked = _check_abi(cfg, 333)
    for k in ("pred", "dy"):
        check_close(k + " chunked vs resident", chunked[k], resident[k], rtol=TOL)


# ------------------------------------------------------------------------------------------------------- whole models, E = 512
SWEEP = dict(num_blocks=2, dimPosIn=66, dimPosEmb=512, dimPosOut=66, in_nTP=10, out_nTP=25, conv_nChan=1, conv1_kernel_shape=(1, 3),
             conv1_stride=(1, 1), conv1_padding=(0, 1), mode_conv="twice", activation="mish", regularization=0.1, use_se=True, r_se=8,
             encoder_n_harmonic_functions=0, encoder_omega0=0)
MODELS = {
    "sweep_dropout": SWEEP,
    "default_encoder_harmonic64": dict(SWEEP, regularization=0, encoder_n_harmonic_functions=64, encoder_omega0=0.1),
    "c8_bn_once": dict(SWEEP, conv_nChan=8, regularization=-1.0, mode_conv="once", conv1_kernel_shape=(5, 9), conv1_padding=None,
                       num_blocks=1),
}


@pytest.mark.parametrize("case", sorted(MODELS))
def test_model_at_e512_vs_oracle(case):
    cfg = MODELS[case]
    model, params = _build(cfg, seed=11)
    model.train()
    x, gt = synthetic_pose_windows(6, 10, 25, cfg["dimPosIn"], scale="amass", seed=5)
    masks = MK.conv_masks(cfg, len(x), 11, step=0) if cfg.get("regularization", 0) > 0 else None
    got = _run(model, x, gt)
    o32, o64 = _oracles(cfg, params, x, gt, masks)
    _compare(got, o32, o64, params)


def test_c8_bn_model_at_e512_tf32():
    cfg = MODELS["c8_bn_once"]
    model, params = _build(cfg, seed=11)
    model.set_precision("tf32")
    model.train()
    x, gt = synthetic_pose_windows(6, 10, 25, cfg["dimPosIn"], scale="amass", seed=5)
    pred, loss, grads, dx = _run(model, x, gt)
    o32, o64 = _oracles(cfg, params, x, gt)
    check_close("pred", pred, o32[0], o64[0], rtol=2e-3)
    floor = 5e-6 * grad_scale(o32[2])
    for k in O.trainable_keys(params):
        check_close("grad " + k, grads[k], o32[2][k], o64[2][k], rtol=2e-3, atol=floor * 50)


def test_trainstep_graph_vs_eager_at_e512():
    from motionmixerconv_b200.train import TrainStep
    cfg = dict(SWEEP, regularization=0)
    x, gt = synthetic_pose_windows(64, 10, 25, 66, scale="amass", seed=9)
    x, gt = torch.from_numpy(x).cuda(), torch.from_numpy(gt).cuda()
    out = []
    for graph in (True, False):
        model, _ = _build(cfg, seed=2)
        ts = TrainStep(model.train(), lr=1e-3, weight_decay=1e-5, use_cuda_graph=graph)
        losses = [float(ts.step(x, gt)) for _ in range(3)]
        torch.cuda.synchronize()
        out.append((losses, torch.cat([p.detach().flatten() for p in model.parameters()]).cpu()))
        if graph:
            ts.release_graphs()
    (la, pa), (lb, pb) = out
    assert np.allclose(la, lb, rtol=1e-5), (la, lb)
    assert (pa - pb).abs().max().item() <= 1e-5 * pb.abs().max().item()


def test_autograd_and_trainstep_same_calls_at_e512(monkeypatch):
    """As tests/test_gpu_one_path.py: one TrainStep step and one autograd step + FusedAdam make the same C ABI calls."""
    from motionmixerconv_b200.functional import mpjpe_error
    from motionmixerconv_b200.train import FusedAdam, TrainStep
    from tests import test_gpu_one_path as OP
    rec = OP._Recorder(OP.L.load())
    monkeypatch.setattr(OP.L, "_lib", rec)
    cfg = dict(SWEEP, regularization=0)
    x, gt = OP._data("conv", cfg)
    m_ts, m_ag = OP._model("conv", cfg, None), OP._model("conv", cfg, None)
    ts = TrainStep(m_ts, lr=1e-3, weight_decay=1e-5, use_cuda_graph=False)
    opt = FusedAdam(m_ag.parameters(), lr=1e-3, weight_decay=1e-5)
    sa, loss_a = OP._record(rec, lambda: float(ts.step(x, gt)))

    def autograd_step():
        opt.zero_grad(set_to_none=True)
        loss = mpjpe_error(m_ag(x), gt)
        loss.backward()
        opt.step()
        return float(loss)
    sb, loss_b = OP._record(rec, autograd_step)
    OP._same_calls(sa, sb)
    assert any(c[0] == "mmx_conv_head_bwd" for c in sa)
    assert loss_a == pytest.approx(loss_b, rel=1e-5)
