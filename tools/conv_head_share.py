"""Kernel times of the ConvMixer output head (forward, backward) in a training step, and their share of the step's kernel time.

    python tools/conv_head_share.py            # env: HEAD_E=256,512 (embedding widths), HEAD_B=16384 (batch), HEAD_STEPS=5

The sweep's ConvMixer configuration (tools/sweep.py) at each width; eager TrainStep steps under torch.profiler (CUDA
activities), after two warm-up steps.  One JSON line per width, with the card's name and power limit.
"""
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from motionmixerconv_b200.conv_mixer_model import ConvMixer  # noqa: E402
from motionmixerconv_b200.train import TrainStep  # noqa: E402


def conv_cfg(E):   # tools/sweep.py conv_cfg
    return dict(num_blocks=4, dimPosIn=66, dimPosEmb=E, dimPosOut=66, in_nTP=10, out_nTP=25, conv_nChan=1, conv1_kernel_shape=(1, 3),
                conv1_stride=(1, 1), conv1_padding=(0, 1), mode_conv="twice", activation="mish", regularization=0.1, use_se=True, r_se=8,
                encoder_n_harmonic_functions=0, encoder_omega0=0)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else torch.cuda.get_device_name()


def kind(name):
    if "HeadFwd" in name:
        return "head_fwd"
    if "HeadBwd" in name:
        return "head_bwd"
    return "other"


def main():
    B, steps = int(os.environ.get("HEAD_B", "16384")), int(os.environ.get("HEAD_STEPS", "5"))
    for E in [int(v) for v in os.environ.get("HEAD_E", "256,512").split(",")]:
        torch.manual_seed(0)
        model = ConvMixer(**conv_cfg(E)).cuda().train()
        ts = TrainStep(model, lr=1e-3, weight_decay=1e-5, use_cuda_graph=False)
        x = torch.randn(B, 10, 66, device="cuda") * 0.3
        gt = torch.randn(B, 25, 66, device="cuda") * 300
        for _ in range(2):
            ts.step(x, gt)
        torch.cuda.synchronize()
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            for _ in range(steps):
                ts.step(x, gt)
            torch.cuda.synchronize()
        us = {"head_fwd": 0.0, "head_bwd": 0.0, "other": 0.0}
        names = {}
        for ev in prof.key_averages():
            t = ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total
            if t <= 0:
                continue
            k = kind(ev.key)
            us[k] += t / steps
            if k != "other":
                names[k] = ev.key[:120]
        total = sum(us.values())
        print(json.dumps({"E": E, "batch": B, "card": card(), "head_fwd_us": us["head_fwd"], "head_bwd_us": us["head_bwd"],
                          "step_kernel_us": total, "head_share": (us["head_fwd"] + us["head_bwd"]) / total, "kernels": names,
                          "basis": "torch.profiler device time per eager TrainStep step, mean of %d steps" % steps}), flush=True)
        del ts, model


if __name__ == "__main__":
    main()
