"""Checkpoint / wire format (SURVEY §8 f4): ``torch.save(model.state_dict())`` files are interchangeable with the REAL reference
modules in both directions (strict), incl. the aliased ``se2.*`` keys, BatchNorm buffers and ``encoder.frequencies``; and a
TrainStep run resumes bit-compatibly from (model.state_dict(), TrainStep.state_dict()).
The reference side is the state_dict the reference modules themselves wrote into the golden fixtures (tests/golden/make_golden.py:
the unmodified reference module built after ``torch.manual_seed(0)``, its ``state_dict()`` stored entry by entry, in order)."""
import io

import numpy as np
import pytest
import torch

from tests.golden_util import Golden, golden_cases


def _roundtrip(sd):
    buf = io.BytesIO()
    torch.save(sd, buf)
    buf.seek(0)
    return torch.load(buf)


def _ours(g):
    from motionmixerconv_b200.conv_mixer_model import ConvMixer
    from motionmixerconv_b200.mlp_mixer import MlpMixer
    return (MlpMixer if g.family == "mlp" else ConvMixer)(**g.cfg)


def _reference_state_dict(g):
    """What the reference module's ``state_dict()`` held: keys in its order, shapes, dtypes and values."""
    return {k: torch.from_numpy(np.array(v)) for k, v in g.params.items()}


def _check_both_ways(ours, sd_r):
    sd_o = ours.state_dict()
    assert list(sd_o.keys()) == list(sd_r.keys())
    assert [tuple(v.shape) for v in sd_o.values()] == [tuple(v.shape) for v in sd_r.values()]
    assert [v.dtype for v in sd_o.values()] == [v.dtype for v in sd_r.values()]
    # product checkpoint -> reference module: its strict load_state_dict needs exactly these keys and shapes, and the values arrive
    ck = _roundtrip(sd_o)
    assert list(ck.keys()) == list(sd_r.keys())
    for k, v in ck.items():
        assert tuple(v.shape) == tuple(sd_r[k].shape) and v.dtype == sd_r[k].dtype and torch.equal(v, sd_o[k]), k
    # reference checkpoint -> product module (strict); parameters moved so that the load is visible (aliases move together)
    params = {n for n, _ in ours.named_parameters(remove_duplicate=False)}
    sd_r = {k: v + 1.0 if k in params else v for k, v in sd_r.items()}
    ours.load_state_dict(_roundtrip(sd_r), strict=True)
    for k, v in ours.state_dict().items():
        assert torch.equal(v, sd_r[k]), k


def test_mlpmixer_checkpoints_interchange_with_the_reference_module():
    for case in golden_cases("mlp"):
        g = Golden(case)
        torch.manual_seed(1)
        _check_both_ways(_ours(g), _reference_state_dict(g))


@pytest.mark.parametrize("case", golden_cases("conv"))
def test_convmixer_checkpoints_interchange_with_the_reference_module(case):
    g = Golden(case)
    torch.manual_seed(1)
    ours = _ours(g)
    _check_both_ways(ours, _reference_state_dict(g))
    if g.cfg["use_se"] and g.cfg["mode_conv"] == "twice":
        sd = ours.state_dict()
        assert sd["Mixer_Block.0.se2.excitationBlock.0.weight"].data_ptr() == sd["Mixer_Block.0.se.excitationBlock.0.weight"].data_ptr()


def test_same_seed_gives_the_reference_modules_initial_weights():
    for case in golden_cases():
        g = Golden(case)
        torch.manual_seed(0)            # the seed the fixture's reference module was built with
        a = _ours(g).state_dict()
        b = _reference_state_dict(g)
        assert list(a.keys()) == list(b.keys()), case
        assert all(torch.equal(a[k], b[k]) for k in b), case


@pytest.mark.gpu
def test_trainstep_resumes_from_a_checkpoint():
    """3 steps, save (model + optimiser state) through torch.save, load into fresh objects, 2 more steps == 5 uninterrupted."""
    from motionmixerconv_b200.mlp_mixer import MlpMixer
    from motionmixerconv_b200.train import TrainStep
    g = Golden("mlp_k2")
    cfg = dict(g.cfg, regularization=0)

    def fresh():
        m = MlpMixer(**cfg)
        m.load_state_dict({k: torch.from_numpy(np.asarray(v)) for k, v in g.params.items()}, strict=True)
        return m.cuda().train()

    x, gt = torch.from_numpy(g.x).cuda(), torch.from_numpy(g.gt).cuda()
    a = TrainStep(fresh(), lr=1e-3, weight_decay=1e-5)
    for _ in range(5):
        a.step(x, gt)
    b = TrainStep(fresh(), lr=1e-3, weight_decay=1e-5)
    for _ in range(3):
        b.step(x, gt)
    ck = _roundtrip({"model": b.model.state_dict(), "optim": b.state_dict()})
    assert ck["optim"]["step"] == 3 and set(ck["optim"]["exp_avg"]) == {n for n, _ in b.model.named_parameters()}
    m2 = MlpMixer(**cfg)
    m2.load_state_dict(ck["model"], strict=True)
    c = TrainStep(m2.cuda().train(), lr=1e-3, weight_decay=1e-5)
    c.load_state_dict(ck["optim"])
    for _ in range(2):
        c.step(x, gt)
    assert c.steps_done == 5
    # Adam normalises every gradient to ~lr per step, so an element whose gradient is rounding noise (order of the REDs) may move
    # differently: count elements that disagree by more than 3 % of the 5e-3 the weights travelled in 5 steps
    bad = tot = 0
    for (k, va), vc in zip(a.model.state_dict().items(), c.model.state_dict().values()):
        bad += int(((va - vc).abs() > 0.03 * 5e-3).sum())
        tot += va.numel()
    assert bad / tot <= 0.005, (bad, tot)
    # and resuming WITHOUT the optimiser state is measurably different (the test would not notice a no-op load otherwise)
    d = TrainStep(fresh(), lr=1e-3, weight_decay=1e-5)
    d.model.load_state_dict(ck["model"], strict=True)
    for _ in range(2):
        d.step(x, gt)
    worse = sum(int(((va - vd).abs() > 0.03 * 5e-3).sum()) for va, vd in zip(a.model.state_dict().values(), d.model.state_dict().values()))
    assert worse > 10 * max(bad, 1)
