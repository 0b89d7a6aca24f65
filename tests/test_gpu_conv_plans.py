"""The fused fp32 ConvMixerBlock kernels (csrc/mmx_conv.cuh, the BatchNorm passes of csrc/mmx_conv_io.cuh) at batches where
every CTA of every pass runs several tiles, against the oracle: the Optuna cell (C = 8, E = 192, 5x5) at its default plans,
whose backward streams X / dY from global memory; every fused fixture with the tile and the backward's input variant forced
(MMX_CONV_S_FWD / MMX_CONV_S_BWD, MMX_CONV_X_GLOBAL); and the BatchNorm ConvMixer and MlpMixer at 16K - 66K sequences, where
the per-CTA accumulators of the batch sums run over ~30 - 110 tiles before they are flushed.

The plan of each pass (tile S, shared memory, grid) is recomputed here from mmx_conv_half_plan and the launch layer's grid
formulas (half_plans), and every test asserts what it claims to cover: each pass runs >= 3 tiles per CTA, the half is routed
to the fused kernels, and the backward is streamed or resident as stated.

The batches are the replicated and sparse constructions of tests/test_gpu_large_batch.py.  With BatchNorm the replicated
batch x[i] = base[i % P] stays exact when B is a multiple of P: every base sequence appears equally often, so the batch
statistics of the whole batch are those of the base set.  Only the running variance differs (nn.BatchNorm updates it with
the unbiased variance over the elements of the batch); expected_running_var derives it from the base-set update.  The
sparse construction does not hold with BatchNorm (the batch means couple dx across sequences) and is used without it.
test_batchnorm_replicated_construction_is_exact checks this on the CPU with the fp64 oracle.

Bar: that of tests/test_gpu_conv.py, fp32, 1e-5 relative per tensor against the fp32 oracle with the fp64 oracle as the
truth of check_close's noise clause.
"""
import collections
import contextlib
import ctypes as C
import os

import numpy as np
import pytest
import torch

from oracle import mixer_np as O
from oracle import mixer_torch as MT
from tests import masks_np as MK
from tests.golden_util import Golden, check_close, grad_scale
from tests.synthetic import synthetic_pose_windows
from tests.test_gpu_large_batch import P, _check_replicated, _check_sparse, _replicate, check_rows, mlp_cfg, replicated_oracle

TOL = 1e-5
FLOOR = 5e-6                                          # gradient floor, x grad_scale
ZERO_GRAD_SLACK = {"encoder.channelUpscaling.bias": 50}
MIN_TILES = 3                                         # tiles every CTA of every covered pass runs
CONV_TILE_ELEMS = 8192                                # kConvTileElems (csrc/mmx_conv_host.cuh)
K_PARTS = 8                                           # kParts (csrc/mmx_mlp.cuh)
DTYPES = (np.float32, np.float64)

# the Optuna grid's production cell (C = 8, E = 192, 5x5, BatchNorm or not)
OPTUNA = dict(num_blocks=2, dimPosIn=33, dimPosEmb=192, dimPosOut=33, in_nTP=10, out_nTP=10, conv_nChan=8, conv1_kernel_shape=(5, 5),
              activation="mish", use_se=True, r_se=8, encoder_n_harmonic_functions=0, encoder_omega0=0)
# padded channels in the CP = 8 instantiation (C = 5), E % 4 != 0 with an odd row pitch (E = 37)
SYNTH_C5_E37 = dict(num_blocks=2, dimPosIn=33, dimPosEmb=37, dimPosOut=33, in_nTP=10, out_nTP=10, conv_nChan=5, conv1_kernel_shape=(3, 3),
                    mode_conv="twice", activation="gelu", regularization=0, use_se=True, r_se=4, use_max_pooling=False,
                    encoder_n_harmonic_functions=0, encoder_omega0=0)


# ------------------------------------------------------------------------------------------ plan arithmetic
Plan = collections.namedtuple("Plan", "where name S smem grid tiles per_cta streamed")


def balanced_grid(ntiles, max_ctas):
    """balanced_grid (csrc/mmx_launch.cuh)."""
    if ntiles <= max_ctas:
        return max(ntiles, 1)
    waves = -(-ntiles // max_ctas)
    return -(-ntiles // waves)


def tile_grid(B, S, smem, sms, optin):
    """tile_grid (csrc/mmx_launch.cuh): as many CTAs as fit the SMs (at most 8 each), balanced over the tiles."""
    return balanced_grid(-(-B // S), sms * max(1, min(8, (optin + 1024) // (smem + 1024))))


def bn_pass_smem(C_, T, E, rr, S):
    """bn_pass_smem (csrc/mmx_conv_io.cuh), bytes."""
    rr, ST = max(rr, 1), S * T
    sizes = [rr * T, T * rr, ST * C_ * K_PARTS, ST * C_ * K_PARTS, ST, ST, S * rr, ST, S * rr, ST, rr * T, T * rr, 16, 32]
    return 4 * sum(-(-n // 4) * 4 for n in sizes)


@contextlib.contextmanager
def env(**kv):
    old = {k: os.environ.get(k) for k in kv}
    os.environ.update({k: str(v) for k, v in kv.items()})
    try:
        yield
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def halves(mb):
    return (0, 1) if mb.mode_conv == "twice" else (0,)


def half_desc(mb, half, B, training=True):
    """The half's descriptor as functional.conv_half_fits / ConvHalf build it."""
    from motionmixerconv_b200 import functional as F_
    m = mb.half_meta(half)
    return F_.conv_half_desc(B, mb.conv_nChan, mb.in_nTP, mb.dimPosEmb, *m[:6], training, *m[7:])


def half_plans(lib, mb, half, B, sms, optin, training=True):
    """The fused passes one ConvMixerBlock half launches at batch B: the descriptor as functional.conv_half_fits / ConvHalf
    build it, S and shared memory from mmx_conv_half_plan, the grid from tile_grid (convolution passes) or plan_bn_pass
    (csrc/mmx_api_conv_fwd.cu: BatchNorm apply and bwd1).  ``streamed`` (backward passes): the X / dY rows are read from
    global memory, i.e. the plan is the same with MMX_CONV_X_GLOBAL=1."""
    Cn, T, E = mb.conv_nChan, mb.in_nTP, mb.dimPosEmb
    m = mb.half_meta(half)
    desc = half_desc(mb, half, B, training)

    def conv(bwd):
        S, smem = C.c_int(0), C.c_int(0)
        assert lib.mmx_conv_half_plan(C.byref(desc), int(bwd), C.byref(S), C.byref(smem)) == 0, lib.mmx_last_error()
        return S.value, smem.value

    def conv_row(name, bwd):
        S, smem = conv(bwd)
        streamed = None
        if bwd:
            with env(MMX_CONV_X_GLOBAL=1):
                hook = conv(True)
            streamed = hook == (S, smem)
            assert streamed or hook[1] < smem, (hook, smem)
        grid = tile_grid(B, S, smem, sms, optin)
        tiles = -(-B // S)
        return Plan((mb.block_index, half), name, S, smem, grid, tiles, tiles // grid, streamed)

    def bn_row(name):
        S = min(B, max(1, CONV_TILE_ELEMS // (Cn * T * E)))
        tiles = -(-B // S)
        grid = balanced_grid(tiles, 4 * sms)
        return Plan((mb.block_index, half), name, S, bn_pass_smem(Cn, T, E, m[2], S), grid, tiles, tiles // grid, None)

    if mb.regularization != -1.0:
        return [conv_row("fwd", False)] + ([conv_row("bwd", True)] if training else [])
    if not training:
        return [conv_row("eval fwd", False)]
    return [conv_row("bn stats", False), bn_row("bn apply"), bn_row("bn bwd1"), conv_row("bn bwd2", True)]


# the passes whose tile MMX_CONV_S_FWD / MMX_CONV_S_BWD force (the BatchNorm apply and bwd1 passes have their own tile)
HOOKED = ("fwd", "bwd", "bn stats", "bn bwd2")


def model_plans(lib, model, B, sms, optin, training=True):
    return [p for mb in model.Mixer_Block for h in halves(mb) for p in half_plans(lib, mb, h, B, sms, optin, training)]


def covers(plans, min_tiles=MIN_TILES):
    return all(p.per_cta >= min_tiles for p in plans)


def report(test, B, plans):
    """One line per pass: the rows of the plan table."""
    for p in plans:
        print("PLAN %s B=%d block=%d half=%d %-9s S=%d smem=%d grid=%d tiles=%d tiles/CTA>=%d %s" % (
            test, B, p.where[0], p.where[1], p.name, p.S, p.smem, p.grid, p.tiles, p.per_cta,
            "" if p.streamed is None else "streamed" if p.streamed else "resident"))


# ------------------------------------------------------------------------------------------ BatchNorm running statistics
def bn_elems_per_seq(family, cfg):
    """prefix of each BatchNorm layer -> elements per channel that one sequence contributes (its batch count is B x this)."""
    out = {}
    for i in range(cfg["num_blocks"]):
        pre = "Mixer_Block.%d" % i
        if family == "conv":
            for cb in ("conv1", "conv2") if cfg.get("mode_conv", "twice") == "twice" else ("conv1",):
                out["%s.%s.reg" % (pre, cb)] = cfg["in_nTP"] * cfg["dimPosEmb"]
        else:       # BatchNorm1d on [B, channels, L]: normalised over B x L
            out[pre + ".mlp_block_token_mixing.reg1"] = cfg["tokens_mlp_dim"]
            out[pre + ".mlp_block_token_mixing.reg2"] = cfg["seq_len"]
            out[pre + ".mlp_block_channel_mixing.reg1"] = cfg["channels_mlp_dim"]
            out[pre + ".mlp_block_channel_mixing.reg2"] = cfg["hidden_dim"]
    return out


def expected_running_var(rv_base, rv0, n_base, n_batch, m=O.BN_MOMENTUM):
    """Running variance after one update on the whole replicated batch, from the update the oracle made on the base set:
    the biased batch variance is recovered from the base-set update and re-weighted with the batch's n / (n - 1)."""
    var_b = (rv_base - (1 - m) * rv0) / m * (n_base - 1) / n_base
    return (1 - m) * rv0 + m * var_b * n_batch / (n_batch - 1)


def expected_running_stats(family, cfg, params0, updated, B):
    """running_mean / running_var the model must hold after one training forward on the replicated batch of B = k x P rows,
    ``updated``: the fp64 oracle's parameters after its forward on the P base sequences."""
    want = {}
    for pre, per_seq in bn_elems_per_seq(family, cfg).items():
        want[pre + ".running_mean"] = updated[pre + ".running_mean"]
        want[pre + ".running_var"] = expected_running_var(updated[pre + ".running_var"], params0[pre + ".running_var"].astype(np.float64),
                                                          P * per_seq, B * per_seq)
    return want


def check_running_stats(model, family, cfg, params0, updated, B):
    sd = {k: v.detach().cpu().numpy() for k, v in model.state_dict().items()}
    want = expected_running_stats(family, cfg, params0, updated, B)
    assert want
    for k, v in want.items():
        np.testing.assert_allclose(sd[k], v, rtol=1e-5, atol=1e-7, err_msg=k)
    for pre in bn_elems_per_seq(family, cfg):
        assert int(sd[pre + ".num_batches_tracked"]) == int(params0[pre + ".num_batches_tracked"]) + 1, pre
    return sd


# ------------------------------------------------------------------------------------------ CPU: the constructions and the planner
def _small_bn_cfgs():
    conv = dict(num_blocks=2, dimPosIn=6, dimPosEmb=12, dimPosOut=6, in_nTP=6, out_nTP=4, conv_nChan=3, conv1_kernel_shape=(3, 3),
                mode_conv="twice", activation="mish", regularization=-1.0, use_se=True, r_se=2, use_max_pooling=False,
                encoder_n_harmonic_functions=0, encoder_omega0=0)
    return {"conv": (conv, 6, 6), "mlp": (mlp_cfg(12, 10, num_blocks=2, regularization=-1.0), 10, 66)}


@pytest.mark.parametrize("family", ["conv", "mlp"])
def test_batchnorm_replicated_construction_is_exact(family):
    """CPU, fp64 oracle, P = 7, B = 3 P: the replicated-batch oracle with BatchNorm equals the oracle of the whole batch (pred,
    loss, dx, every gradient, running mean), and expected_running_var gives the whole batch's running variance."""
    cfg, T, D = _small_bn_cfgs()[family]
    n, B = 7, 21
    params = {k: v.numpy().copy() for k, v in MT.random_params(family, cfg, seed=5).items()}
    rng = np.random.default_rng(8)
    for k in params:       # non-trivial initial running statistics: the correction must not rely on rv0 = 1
        if k.endswith("running_var"):
            params[k] = (0.5 + rng.random(params[k].shape)).astype(np.float32)
        if k.endswith("running_mean"):
            params[k] = (0.3 * rng.standard_normal(params[k].shape)).astype(np.float32)
    Orc = O.ConvMixerOracle if family == "conv" else O.MlpMixerOracle
    To = cfg["out_nTP"] if family == "conv" else cfg["pred_len"]
    xb, gtb = synthetic_pose_windows(n, T, To, D, scale="amass", seed=2)
    x, gt = xb[np.arange(B) % n], gtb[np.arange(B) % n]

    full = Orc(cfg, params, dtype=np.float64)
    pred = full.forward(x, training=True)
    loss, dp = O.mpjpe(pred, gt.astype(np.float64))
    grads, dx = full.backward(dp)
    base = Orc(cfg, params, dtype=np.float64)
    rep = replicated_oracle(base, xb, gtb, B)

    def close(a, b, scale=0.0):
        return float(np.abs(a - b).max()) <= 1e-12 * float(np.abs(b).max()) + 1e-14 * scale

    assert close(rep.pred[np.arange(B) % n], pred)
    assert abs(rep.loss - float(loss)) < 1e-12 * float(loss)
    assert close(rep.dx[np.arange(B) % n], dx)
    for k, g in grads.items():
        assert close(rep.grads[k], g, grad_scale(grads)), k
    per_seq = bn_elems_per_seq(family, cfg)
    assert len(per_seq) == sum(k.endswith("running_var") for k in params)
    naive = 0.0
    for pre, L_ in per_seq.items():
        assert close(base.p[pre + ".running_mean"], full.p[pre + ".running_mean"]), pre
        rv = expected_running_var(base.p[pre + ".running_var"], params[pre + ".running_var"].astype(np.float64), n * L_, B * L_)
        assert close(rv, full.p[pre + ".running_var"]), pre
        naive = max(naive, float(np.abs(base.p[pre + ".running_var"] - full.p[pre + ".running_var"]).max()))
    assert naive > 1e-9          # without the correction the running variance would differ


def _cpu_model(cfg, params=None, seed=3):
    from motionmixerconv_b200.conv_mixer_model import ConvMixer
    torch.manual_seed(seed)
    m = ConvMixer(**cfg)
    if params is not None:
        m.load_state_dict({k: torch.from_numpy(np.asarray(v)) for k, v in params.items()}, strict=True)
    return m.train()


B200_SMS, B200_OPTIN = 148, 227 * 1024


def test_planner_claims_on_the_emulator_build():
    """The planner facts the GPU tests below rest on, on the CPU build of the launch layer (same planner, same 227 KB budget),
    with the B200's 148 SMs for the grids: the Optuna 5x5 cell's default backward is the streamed plan at both batches used
    below; the forced tile takes effect; MMX_CONV_X_GLOBAL=1 lowers the backward's shared memory where the resident plan fits;
    and each forced configuration's batch gives every pass >= 3 tiles per CTA under both input variants."""
    from tests.emu.harness import emu
    lib = emu()
    for mode, reg, B in (("once", -1.0, 16 * P), ("twice", 0, 16 * P + 7), ("twice", 0.1, None)):
        model = _cpu_model(dict(OPTUNA, mode_conv=mode, regularization=reg))
        with env(MMX_CONV_X_GLOBAL=0, MMX_CONV_S_FWD=0, MMX_CONV_S_BWD=0):
            B = B or dropout_batch(lib, model, B200_SMS, B200_OPTIN)
            plans = model_plans(lib, model, B, B200_SMS, B200_OPTIN)
        bwd = [p for p in plans if p.streamed is not None]
        assert bwd and all(p.streamed and p.S == 1 for p in bwd), plans
        assert covers(plans), plans
    for name in FORCED:
        cfg, params = forced_config(name)
        model = _cpu_model(cfg, params)
        S, B = forced_plan(lib, model, B200_SMS, B200_OPTIN)
        for xg in (0, 1):
            with env(MMX_CONV_X_GLOBAL=xg, MMX_CONV_S_FWD=S, MMX_CONV_S_BWD=S):
                plans = model_plans(lib, model, B, B200_SMS, B200_OPTIN)
            assert covers(plans), (name, xg, plans)
            assert S == FORCED_S[name] and all(p.S == S for p in plans if p.name in HOOKED), (name, xg, plans)
            assert all(p.streamed == bool(xg) for p in plans if p.streamed is not None), (name, xg, plans)


# ------------------------------------------------------------------------------------------ the forced plans
FORCED = ["conv_k1", "conv_harm64", "conv_evenk", "conv_k3", "conv_once_se", "conv_once_nose", "conv_k3_bn", "synth_c5_e37"]
# the tile forced_plan picks: 2 everywhere but conv_k3 (C = 4, E = 192, 5x9 / 9x5), whose resident backward fits one sequence only
FORCED_S = dict({n: 2 for n in FORCED}, conv_k3=1)


def forced_config(name):
    if name == "synth_c5_e37":
        cfg = SYNTH_C5_E37
        return cfg, {k: v.numpy().copy() for k, v in MT.random_params("conv", cfg, seed=12).items()}
    g = Golden(name)
    return g.cfg, g.params


def forced_plan(lib, model, sms, optin):
    """The forced tile (2 where the planner serves every half at 2 with the backward's X / dY resident, else 1) and the batch:
    the smallest multiple of P (plus a ragged remainder without BatchNorm) at which every pass runs >= 3 tiles per CTA under
    both input variants."""
    def plans(S, B, xg):
        with env(MMX_CONV_X_GLOBAL=xg, MMX_CONV_S_FWD=S, MMX_CONV_S_BWD=S):
            return model_plans(lib, model, B, sms, optin)

    def served(S):
        with env(MMX_CONV_X_GLOBAL=0, MMX_CONV_S_FWD=S, MMX_CONV_S_BWD=S):
            return all(lib.mmx_conv_half_plan(C.byref(half_desc(mb, h, 4 * P)), bwd, None, None) == 0
                       for mb in model.Mixer_Block for h in halves(mb) for bwd in (0, 1))
    S = 2 if served(2) and all(p.streamed is not True for p in plans(2, 4 * P, 0)) else 1
    assert served(S)
    assert all(p.S == S and p.streamed is not True for p in plans(S, 4 * P, 0) if p.name in HOOKED)
    bn = any(mb.regularization == -1.0 for mb in model.Mixer_Block)
    for k in range(1, 65):
        B = k * P if bn else k * P + 5 + int((k * P + 5) % S == 0)
        if all(covers(plans(S, B, xg)) for xg in (0, 1)):
            return S, B
    raise AssertionError("no batch up to 64 P gives every pass %d tiles per CTA" % MIN_TILES)


def dropout_batch(lib, model, sms, optin):
    """The smallest B = 3 x SMs x k + 5 (a ragged last wave) at which every pass runs >= 3 tiles per CTA."""
    return next(B for B in (MIN_TILES * sms * k + 5 for k in range(1, 9)) if covers(model_plans(lib, model, B, sms, optin)))


# ------------------------------------------------------------------------------------------ GPU side
def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _optin():
    return torch.cuda.get_device_properties(0).shared_memory_per_block_optin


def _gpu_model(cfg, params):
    from motionmixerconv_b200.conv_mixer_model import ConvMixer
    m = ConvMixer(**cfg)
    m.load_state_dict({k: torch.from_numpy(np.asarray(v)) for k, v in params.items()}, strict=True)
    return m.cuda().train()


def _fresh_params(cfg, seed):
    return {k: v.detach().numpy().copy() for k, v in _cpu_model(cfg, seed=seed).state_dict().items()}


def _assert_fused_plans(test, model, B, training=True):
    """Every half on the fused kernels, every pass >= 3 tiles per CTA; returns the plans (printed as table rows)."""
    from motionmixerconv_b200 import _lib as L
    assert not any(mb.uses_large_path(h, B) for mb in model.Mixer_Block for h in halves(mb)), "a half left the fused kernels"
    plans = model_plans(L.load(), model, B, _sms(), _optin(), training)
    report(test, B, plans)
    assert covers(plans), plans
    return plans


def _grad_atol(k):
    return ZERO_GRAD_SLACK.get(k, 1)


Oracle = collections.namedtuple("Oracle", "cfg params xb gtb B reps updated")


def _replicated_oracles(family, cfg, params, B, seed):
    """fp32 and fp64 replicated-batch oracles of the batch x[i] = xb[i % P] and the fp64 oracle's parameters after its forward
    (BatchNorm running statistics of the base set)."""
    if family == "conv":
        xb, gtb = synthetic_pose_windows(P, cfg["in_nTP"], cfg["out_nTP"], cfg["dimPosIn"], scale="amass", seed=seed)
        Orc = O.ConvMixerOracle
    else:
        xb, gtb = synthetic_pose_windows(P, cfg["seq_len"], cfg["pred_len"], cfg["input_size"], scale="amass", seed=seed)
        Orc = O.MlpMixerOracle
    reps, updated = [], None
    for dt in DTYPES:
        o = Orc(cfg, params, dtype=dt)
        reps.append(replicated_oracle(o, xb, gtb, B))
        updated = o.p
    return Oracle(cfg, params, xb, gtb, B, reps, updated)


def _check_eval_rows(model, orc, family, sd):
    """Eval forward of the replicated batch (the fused forward with the constant BatchNorm affine) against the oracle's eval
    forward with the model's updated running statistics."""
    Orc = O.ConvMixerOracle if family == "conv" else O.MlpMixerOracle
    p = {**orc.params, **{k: sd[k] for k in orc.params if "running_" in k or "num_batches" in k}}
    want, truth = (Orc(orc.cfg, p, dtype=dt).forward(orc.xb, training=False) for dt in DTYPES)
    model.eval()
    with torch.no_grad():
        pe = model(_replicate(orc.xb, orc.B))
    torch.cuda.synchronize()
    check_rows("pred_eval", pe, want, truth, rtol=TOL)


# ---- the Optuna cell at its default plans
@pytest.fixture(scope="module")
def optuna_bn_oracle():
    cfg = dict(OPTUNA, mode_conv="once", regularization=-1.0)
    return _replicated_oracles("conv", cfg, _fresh_params(cfg, seed=5), 16 * P, seed=31)


@pytest.mark.gpu
def test_optuna_cell_batchnorm_at_16k(optuna_bn_oracle, monkeypatch):
    """mode "once" + BatchNorm at B = 16 P = 16,496: statistics pass, apply pass, bwd1, bwd2 on the streamed plan and the eval
    forward, each with >= 3 tiles per CTA (the statistics pass ~110); every pred and dx row, the loss, every gradient, the
    running statistics, then the eval forward."""
    for k in ("MMX_CONV_X_GLOBAL", "MMX_CONV_S_FWD", "MMX_CONV_S_BWD"):
        monkeypatch.delenv(k, raising=False)
    orc = optuna_bn_oracle
    model = _gpu_model(orc.cfg, orc.params)
    plans = _assert_fused_plans("optuna_bn_once", model, orc.B)
    assert all(p.streamed for p in plans if p.name == "bn bwd2")
    _assert_fused_plans("optuna_bn_once", model, orc.B, training=False)
    _check_replicated(model, orc.reps, orc.xb, orc.gtb, orc.B, TOL, FLOOR, dx_atol_k=1e-6, grad_atol=_grad_atol)
    sd = check_running_stats(model, "conv", orc.cfg, orc.params, orc.updated, orc.B)
    _check_eval_rows(model, orc, "conv", sd)


@pytest.fixture(scope="module")
def optuna_twice_oracle():
    cfg = dict(OPTUNA, mode_conv="twice", regularization=0)
    return _replicated_oracles("conv", cfg, _fresh_params(cfg, seed=6), 16 * P + 7, seed=32)


@pytest.mark.gpu
def test_optuna_cell_twice_at_16k_ragged(optuna_twice_oracle, monkeypatch):
    """mode "twice" without BatchNorm at B = 16 P + 7, both halves' backward on the streamed plan: the replicated check, then
    the sparse one (dx exactly 0 outside the sequences that carry dpred: a tile that reads another tile's dY from global
    memory shows up there)."""
    for k in ("MMX_CONV_X_GLOBAL", "MMX_CONV_S_FWD", "MMX_CONV_S_BWD"):
        monkeypatch.delenv(k, raising=False)
    orc = optuna_twice_oracle
    model = _gpu_model(orc.cfg, orc.params)
    plans = _assert_fused_plans("optuna_twice", model, orc.B)
    assert all(p.streamed for p in plans if p.name == "bwd") and len(plans) == 8
    _check_replicated(model, orc.reps, orc.xb, orc.gtb, orc.B, TOL, FLOOR, dx_atol_k=1e-6, grad_atol=_grad_atol)
    _check_sparse(model, [O.ConvMixerOracle(orc.cfg, orc.params, dtype=dt) for dt in DTYPES], orc.xb, orc.B, TOL, FLOOR)


@pytest.mark.gpu
def test_optuna_cell_twice_dropout(monkeypatch):
    """mode "twice", dropout 0.1, at the smallest B = 3 x SMs x k + 5 that gives every pass >= 3 tiles per CTA: the full fp64 /
    fp32 oracles with the masks the kernels draw (masks are per sequence: no replicated batch)."""
    from motionmixerconv_b200 import _lib as L
    from motionmixerconv_b200.functional import mpjpe_error
    for k in ("MMX_CONV_X_GLOBAL", "MMX_CONV_S_FWD", "MMX_CONV_S_BWD"):
        monkeypatch.delenv(k, raising=False)
    cfg = dict(OPTUNA, mode_conv="twice", regularization=0.1)
    params = _fresh_params(cfg, seed=7)
    B = dropout_batch(L.load(), _cpu_model(cfg, params), _sms(), _optin())
    x, gt = synthetic_pose_windows(B, 10, 10, 33, scale="amass", seed=33)
    model = _gpu_model(cfg, params)
    plans = _assert_fused_plans("optuna_twice_dropout", model, B)
    assert all(p.streamed for p in plans if p.name == "bwd")
    torch.manual_seed(4321)                                 # the blocks draw their dropout seed from torch.initial_seed()
    xg = torch.from_numpy(x).cuda().requires_grad_(True)
    pred = model(xg)
    loss = mpjpe_error(pred, torch.from_numpy(gt).cuda())
    loss.backward()
    torch.cuda.synchronize()
    masks = MK.conv_masks(cfg, B, 4321, step=0)
    res = []
    for dt in DTYPES:
        o = O.ConvMixerOracle(cfg, params, dtype=dt)
        p = o.forward(x, training=True, masks=masks)
        l, dp = O.mpjpe(p, gt.astype(dt))
        res.append((p, l, *o.backward(dp)))
    (p32, _, g32, dx32), (p64, l64, g64, dx64) = res
    check_close("pred", pred.detach().cpu().numpy(), p32, p64, rtol=TOL)
    assert abs(float(loss.detach()) - float(l64)) <= TOL * abs(float(l64))
    floor = FLOOR * grad_scale(g32)
    grads = {k: p.grad.detach().cpu().numpy() for k, p in model.named_parameters()}
    for k in O.trainable_keys(params):
        if ".se2." in k:
            continue
        check_close("grad " + k, grads[k], g32[k], g64[k], rtol=TOL, atol=floor * _grad_atol(k))
    check_close("dx", xg.grad.cpu().numpy(), dx32, dx64, rtol=TOL, atol=1e-6 * float(np.abs(dx32).max()))


# ---- every fused plan, forced
@pytest.fixture(scope="module")
def forced_oracles():
    from motionmixerconv_b200 import _lib as L
    cache = {}

    def get(name):
        if name not in cache:
            cfg, params = forced_config(name)
            S, B = forced_plan(L.load(), _cpu_model(cfg, params), _sms(), _optin())
            cache[name] = (S, _replicated_oracles("conv", cfg, params, B, seed=40 + FORCED.index(name)))
        return cache[name]
    return get


@pytest.mark.gpu
@pytest.mark.parametrize("name", FORCED)
@pytest.mark.parametrize("xg", [0, 1], ids=["resident", "streamed"])
def test_forced_plan_several_tiles_per_cta(name, xg, forced_oracles, monkeypatch):
    """Tile forced to 2 (1 where 2 does not fit), the backward's X / dY resident or streamed, at the smallest multiple of P
    (plus a ragged remainder without BatchNorm) that gives every pass >= 3 tiles per CTA: on the device, the shared-memory
    accumulators and the cross-CTA flushes that the emulator runs one CTA at a time."""
    S, orc = forced_oracles(name)
    monkeypatch.setenv("MMX_CONV_X_GLOBAL", str(xg))
    monkeypatch.setenv("MMX_CONV_S_FWD", str(S))
    monkeypatch.setenv("MMX_CONV_S_BWD", str(S))
    model = _gpu_model(orc.cfg, orc.params)
    plans = _assert_fused_plans("forced_%s_%s" % (name, "streamed" if xg else "resident"), model, orc.B)
    assert all(p.S == S for p in plans if p.name in HOOKED)
    assert all(p.streamed == bool(xg) for p in plans if p.streamed is not None)
    _check_replicated(model, orc.reps, orc.xb, orc.gtb, orc.B, TOL, FLOOR, dx_atol_k=1e-6, grad_atol=_grad_atol)
    if orc.cfg["regularization"] == -1.0:
        check_running_stats(model, "conv", orc.cfg, orc.params, orc.updated, orc.B)
    else:
        _check_sparse(model, [O.ConvMixerOracle(orc.cfg, orc.params, dtype=dt) for dt in DTYPES], orc.xb, orc.B, TOL, FLOOR)


# ---- the MlpMixer BatchNorm1d chain at a sweep-size batch
@pytest.mark.gpu
def test_mlp_batchnorm_chain_at_66k():
    """K2 widths with BatchNorm1d (H = ch = 50, tok = 20, mish, SE, 2 blocks) at B = 64 P = 65,984: pred and dx rows, every
    gradient, the running statistics and the eval forward."""
    from motionmixerconv_b200 import functional as F_
    from motionmixerconv_b200.mlp_mixer import MlpMixer
    cfg = mlp_cfg(50, 50, num_blocks=2, regularization=-1.0)
    torch.manual_seed(8)
    m = MlpMixer(**cfg)
    params = {k: v.detach().numpy().copy() for k, v in m.state_dict().items()}
    model = m.cuda().set_precision("fp32").train()
    orc = _replicated_oracles("mlp", cfg, params, 64 * P, seed=48)
    for mb in model.Mixer_Block:           # every block runs as the BatchNorm1d stage-kernel chain
        assert [type(r) for r in mb.runners(orc.B, "cuda", False)] == [F_.MlpBnBlock]
    _check_replicated(model, orc.reps, orc.xb, orc.gtb, orc.B, TOL, FLOOR, dx_atol_k=1e-6)
    sd = check_running_stats(model, "mlp", cfg, params, orc.updated, orc.B)
    _check_eval_rows(model, orc, "mlp", sd)
