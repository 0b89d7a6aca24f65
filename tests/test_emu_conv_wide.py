"""CPU: the ConvMixer PoseEncoder and output head at the embedding widths their resident tiles do not hold (E up to 512),
run from the kernel source in the host emulator (tests/emu/harness.py) against the fp32 + fp64 numpy oracle.

A model with num_blocks = 0 is exactly encoder -> head, so the oracle's forward / backward checks those two kernels alone.
MMX_CHEAD_EC forces the chunked head plan and its chunk width, MMX_ENC_HC the split-harmonic encoder chunk and
MMX_ENC_BWD_ROWS the encoder backward's staged frames: that puts the chunk loops, with a ragged last chunk, on small shapes.
"""
import numpy as np
import pytest

from oracle import mixer_np as O
from tests.emu import harness as H
from tests.golden_util import check_close, grad_scale
from tests.synthetic import synthetic_pose_windows

TOL = 1e-5


def _params(cfg, seed):
    from oracle.mixer_torch import random_params
    p = {k: v.numpy().copy() for k, v in random_params("conv", cfg, seed=seed).items()}
    rng = np.random.default_rng(seed)
    E = cfg["dimPosEmb"]
    p["LN.weight"] = (1.0 + 0.3 * rng.standard_normal(E)).astype(np.float32)    # non-trivial dgamma / dbeta paths
    p["LN.bias"] = (0.2 * rng.standard_normal(E)).astype(np.float32)
    return p


def _check(cfg, B, seed=1):
    params = _params(cfg, seed)
    x, _ = synthetic_pose_windows(B, cfg["in_nTP"], cfg["out_nTP"], cfg["dimPosIn"], scale="amass", seed=seed)
    dout = np.random.default_rng(seed + 1).standard_normal((B, cfg["out_nTP"], cfg["dimPosOut"])).astype(np.float32)
    ref = []
    for dt in (np.float32, np.float64):
        o = O.ConvMixerOracle(cfg, params, dtype=dt)
        ref.append((o.forward(x),) + o.backward(dout.astype(dt)))
    (p32, g32, dx32), (p64, g64, dx64) = ref
    m = H.EmuConvMixer(cfg, params, training=True)
    check_close("pred", m.forward(x), p32, p64, rtol=TOL)
    grads, dx = m.backward(dout)
    floor = 5e-6 * grad_scale(g32)
    for k in O.trainable_keys(params):
        check_close("grad " + k, grads[k], g32[k], g64[k], rtol=TOL, atol=floor * (50 if k == "encoder.channelUpscaling.bias" else 1))
    check_close("dx", dx, dx32, dx64, rtol=TOL, atol=1e-6 * float(np.abs(dx32).max()))


def _cfg(**kw):
    base = dict(num_blocks=0, dimPosIn=9, dimPosEmb=30, dimPosOut=11, in_nTP=10, out_nTP=25, conv_nChan=3,
                encoder_n_harmonic_functions=5, encoder_omega0=0.1)
    base.update(kw)
    return base


@pytest.mark.parametrize("C,ec,S,B", [(3, 8, 2, 69), (1, 12, 3, 7), (8, 16, 1, 3)])
def test_emulated_chunked_head_forced(C, ec, S, B, monkeypatch):
    """Chunked head at E = 30: chunks of 8 (ragged last of 6), 12 (last of 6) and 16 (last of 14); B = 69 in tiles of two
    gives 35 tiles on 18 CTAs: two tiles per CTA, the last one ragged."""
    monkeypatch.setenv("MMX_CHEAD_EC", str(ec))
    monkeypatch.setenv("MMX_CHEAD_S_FWD", str(S))
    monkeypatch.setenv("MMX_CHEAD_S_BWD", str(S))
    _check(_cfg(conv_nChan=C), B)


@pytest.mark.parametrize("hc,rows", [(3, 16), (2, 7), (1, 64)])
def test_emulated_split_harmonic_encoder_forced(hc, rows, monkeypatch):
    """Harmonic encoder with Hn = 5 split into chunks of hc harmonics of one input dimension (ragged last segment), and
    the backward's sweep over the frames in steps of `rows` (ragged last step)."""
    monkeypatch.setenv("MMX_ENC_HC", str(hc))
    monkeypatch.setenv("MMX_ENC_BWD_ROWS", str(rows))
    _check(_cfg(), 11)


@pytest.mark.parametrize("C,Hn,E", [(1, 64, 512), (8, 0, 512), (2, 16, 509)])
def test_emulated_wide_embedding_unforced(C, Hn, E):
    """E = 512 (and an odd 509) with the plans chosen by shape: the chunked head, the split-harmonic encoder forward and
    the backward's staged rows picked to fit; the plain (Hn = 0) encoder at E = 512 needs neither."""
    _check(_cfg(conv_nChan=C, encoder_n_harmonic_functions=Hn, dimPosEmb=E, dimPosOut=66), 3)
