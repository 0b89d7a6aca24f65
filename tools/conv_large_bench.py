"""ConvMixer training-step throughput on the reference's Optuna-grid shapes (optuna_search/conv_optuna_main.py:339-342: C = 8,
E = 192, 6 blocks, BatchNorm, 'once'), fused kernels vs the stage-kernel chain, next to the reference modules on the host.
    python tools/conv_large_bench.py            (on a B200)
Environment: B (batch, 256), STEPS (timed steps, 10), PRECISION ("fp32" default | "tf32": ConvMixer.set_precision), WITH_REF."""
import json
import os
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from motionmixerconv_b200.conv_mixer_model import ConvMixer
from motionmixerconv_b200.train import TrainStep
from tests.synthetic import synthetic_pose_windows

B = int(os.environ.get("B", 256))
STEPS = int(os.environ.get("STEPS", 10))
PRECISION = os.environ.get("PRECISION", "fp32")


def cfg_of(kt, kp, mode="once", reg=-1.0, C=8):
    return dict(num_blocks=6, dimPosIn=33, dimPosEmb=192, dimPosOut=33, in_nTP=10, out_nTP=10, conv_nChan=C, conv1_kernel_shape=(kt, kp),
                mode_conv=mode, activation="mish", regularization=reg, use_se=True, r_se=8, encoder_n_harmonic_functions=0, encoder_omega0=0)


def ours(cfg, precision=None):
    torch.manual_seed(0)
    model = ConvMixer(**cfg).cuda().train().set_precision(precision or PRECISION)
    x, gt = synthetic_pose_windows(B, 10, 10, 33, scale="ais", seed=1)
    xs, gts = torch.from_numpy(x).cuda(), torch.from_numpy(gt).cuda()
    ts = TrainStep(model, lr=1e-3, weight_decay=1e-5)
    for _ in range(3):
        ts.step(xs, gts)
    torch.cuda.synchronize()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(STEPS):
        loss = ts.step(xs, gts)
    e.record()
    torch.cuda.synchronize()
    ms = s.elapsed_time(e) / STEPS
    chain = any(mb.uses_large_path(h, B) for mb in model.Mixer_Block for h in ((0, 1) if mb.mode_conv == "twice" else (0,)))
    return ms, chain, float(loss)


def reference(cfg, steps=2):
    from oracle import make_ref
    if not make_ref.available():
        return None
    _, RefConv, mpjpe = make_ref.import_reference()
    torch.manual_seed(0)
    torch.set_num_threads(os.cpu_count() or 1)
    m = RefConv(**cfg).train()
    opt = torch.optim.Adam(m.parameters(), lr=1e-3, weight_decay=1e-5)
    x, gt = synthetic_pose_windows(B, 10, 10, 33, scale="ais", seed=1)
    x, gt = torch.from_numpy(x), torch.from_numpy(gt)

    def step():
        opt.zero_grad()
        l = mpjpe(m(x), gt)
        l.backward()
        opt.step()
    step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    return (time.perf_counter() - t0) / steps * 1e3


def main():
    for kt, kp in ((5, 5), (5, 9), (9, 9), (9, 29), (1, 29)):
        for mode in ("once", "twice"):
            cfg = cfg_of(kt, kp, mode)
            ms, chain, loss = ours(cfg)
            ref_ms = reference(cfg) if os.environ.get("WITH_REF", "1") == "1" and mode == "once" else None
            print(json.dumps({"C": 8, "E": 192, "kernel": [kt, kp], "mode_conv": mode, "B": B, "precision": PRECISION,
                              "path": "stage-kernel chain" if chain else "fused kernels",
                              "ms_per_step": round(ms, 3), "seq_per_s": round(B / ms * 1e3), "loss": round(loss, 4),
                              "reference_cpu_ms": None if ref_ms is None else round(ref_ms, 1),
                              "reference_cpu_seq_per_s": None if ref_ms is None else round(B / ref_ms * 1e3), "cores": os.cpu_count()}), flush=True)


if __name__ == "__main__":
    main()
