"""fp32 vs tcgen05 ("tf32") ConvMixer convolutions on a B200, modes alternated within one process, one JSON line per cell:
  * the card (name, power limit);
  * kernel times (CUDA events) of mmx_conv2d_large_{fwd,wgrad}_prec and the data gradient on the Optuna cells (C = 8, T = 10,
    E = 192, B = 256), with the achieved rate 2 * B * C^2 * kt * kp * T * E / time;
  * training steps of tools/conv_large_bench.py on the Optuna cells (once / twice), and the K3 rollout training (RolloutTrainer
    graph) at B = 256, in fp32 and tf32; in tf32 also with every half forced onto the chain (MMX_CONV_FORCE_LARGE=1), the A/B
    behind the tf32 routing of ConvMixerBlock.uses_large_path.
    python tools/conv_tc5_profile.py OUT.jsonl"""
import ctypes as C
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from motionmixerconv_b200 import _lib as L
from motionmixerconv_b200 import functional as F_

OUT = open(sys.argv[1] if len(sys.argv) > 1 else os.devnull, "w")


def emit(rec):
    line = json.dumps(rec)
    print(line, flush=True)
    OUT.write(line + "\n")
    OUT.flush()


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    emit({"card": q.stdout.strip().splitlines()[0] if q.stdout else "?"})


def events(fn, n):
    fn()
    torch.cuda.synchronize()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(n):
        fn()
    e.record()
    torch.cuda.synchronize()
    return s.elapsed_time(e) / n


def kernels(B=256, Cn=8, T=10, E=192, n=20):
    lib = L.load()
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    g = torch.Generator(device="cuda").manual_seed(0)
    x = torch.randn(B, Cn, T, E, device="cuda", generator=g)
    dz = torch.randn(B, Cn, T, E, device="cuda", generator=g)
    out = torch.empty_like(x)
    p = lambda t: C.c_void_p(t.data_ptr())
    for kt, kp in ((5, 5), (5, 9), (9, 9), (9, 29)):
        d = F_.conv_half_desc(B, Cn, T, E, (kt, kp), ((kt - 1) // 2, (kp - 1) // 2), 0, "gelu", False, False, False, 0, 0.0, 0, 0)
        w = torch.randn(Cn, Cn, kt, kp, device="cuda", generator=g) * 0.05
        b = torch.zeros(Cn, device="cuda")
        dw, db = torch.zeros_like(w), torch.zeros_like(b)
        flop = 2.0 * B * Cn * Cn * kt * kp * T * E
        rec = {"kernel_times": [kt, kp], "B": B, "C": Cn, "T": T, "E": E, "tc5_serves": int(lib.mmx_conv2d_tc5_serves(C.byref(d)))}
        for prec in ("fp32", "tf32", "fp32", "tf32"):
            pr = L.MMX_PREC[prec]
            for name, fn in (("fwd", lambda: lib.mmx_conv2d_large_fwd_prec(C.byref(d), 0, p(x), p(w), p(b), p(out), pr, st)),
                             ("dgrad", lambda: lib.mmx_conv2d_large_fwd_prec(C.byref(d), 1, p(dz), p(w), None, p(out), pr, st)),
                             ("wgrad", lambda: lib.mmx_conv2d_large_wgrad_prec(C.byref(d), p(dz), p(x), p(dw), p(db), pr, st))):
                ms = events(fn, n)
                rec.setdefault(prec, {}).setdefault(name, []).append({"us": round(ms * 1e3, 1), "tflops": round(flop / ms / 1e9, 2)})
        emit(rec)


def train_cells():
    import conv_large_bench as CB
    for kt, kp in ((5, 5), (5, 9), (9, 9), (9, 29)):
        for mode in ("once", "twice"):
            cfg = CB.cfg_of(kt, kp, mode)
            rec = {"train_step": [kt, kp], "mode_conv": mode, "B": CB.B, "C": 8, "E": 192, "steps": CB.STEPS}
            for prec, force in (("fp32", "0"), ("tf32", "0"), ("tf32", "1"), ("fp32", "0"), ("tf32", "0"), ("tf32", "1")):
                os.environ["MMX_CONV_FORCE_LARGE"] = force
                ms, chain, loss = CB.ours(cfg, prec)
                key = prec + ("_forced_chain" if force == "1" else "")
                rec.setdefault(key, []).append({"ms": round(ms, 3), "seq_per_s": round(CB.B / ms * 1e3), "chain": chain, "loss": round(loss, 4)})
            os.environ["MMX_CONV_FORCE_LARGE"] = "0"
            emit(rec)


def k3_rollout(B=256, n=10):
    from argparse import Namespace
    from motionmixerconv_b200.conv_mixer_model import ConvMixer
    from motionmixerconv_b200.rollout import RolloutTrainer
    from tests.synthetic import synthetic_full_windows
    cfg = dict(num_blocks=6, dimPosIn=33, dimPosEmb=192, dimPosOut=33, in_nTP=10, out_nTP=5, conv_nChan=4, conv1_kernel_shape=(5, 9),
               mode_conv="twice", activation="mish", regularization=-1.0, use_se=True, r_se=8, encoder_n_harmonic_functions=0, encoder_omega0=0)
    args = Namespace(input_n_dataset=10, output_n_dataset=25, input_n_model=10, output_n_model=5, step_window=5, loss_type="mpjpe")
    batch = torch.from_numpy(synthetic_full_windows(B, 35, 33, scale="ais", seed=1)).cuda()
    rec = {"k3_rollout_train": "C=4, E=192, k=(5,9)/(9,5), BatchNorm, 6 blocks, 10 -> 25 frames", "B": B}
    for prec, force in (("fp32", "0"), ("tf32", "0"), ("tf32", "1"), ("fp32", "0"), ("tf32", "0"), ("tf32", "1")):
        os.environ["MMX_CONV_FORCE_LARGE"] = force
        torch.manual_seed(0)
        model = ConvMixer(**cfg).cuda().train().set_precision(prec)
        chain = [mb.uses_large_path(h, B) for mb in model.Mixer_Block for h in (0, 1)]
        tr = RolloutTrainer(model, args, list(range(33)), teacher_forcing=False)
        for _ in range(3):
            tr.step(batch)
        ms = events(lambda: tr.step(batch), n)
        key = prec + ("_forced_chain" if force == "1" else "")
        rec.setdefault(key, []).append({"ms": round(ms, 3), "seq_per_s": round(B / ms * 1e3), "halves_on_chain": sum(chain),
                                        "nan": bool(tr.nan_flag)})
        del model, tr
        torch.cuda.empty_cache()
    os.environ["MMX_CONV_FORCE_LARGE"] = "0"
    emit(rec)


if __name__ == "__main__":
    os.environ.setdefault("WITH_REF", "0")
    card()
    kernels()
    train_cells()
    k3_rollout()
    card()
