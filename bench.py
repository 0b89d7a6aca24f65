#!/usr/bin/env python
"""Benchmark of the hot path: train sequences/sec (fwd + MPJPE + bwd + Adam), BASELINE.json's metric.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload k2|k4] [--dump-outputs DIR]

N=1 workload = BASELINE.json configs[1]: MotionMixer MlpMixer with squeeze-excitation, H36M xyz
10 -> 10 frames, batch 4096 per GPU (SURVEY.md §8d "K2": hidden 50, tokens 20, channels 50, 4 blocks,
mish, dropout 0.1, r_se 8).  N>1: the driver launches this file under torchrun; each rank trains on
its own shard of the global batch (weak scaling: 4096 sequences per GPU) with one flat-bucket NCCL
all-reduce per step.  One JSON line is printed by rank 0.

``--dump-outputs DIR`` writes what the timed path computed in its last timed step as ``DIR/<name>.npy`` (see ``step_outputs``).  The
inputs and the initial weights are seeded, so two builds run with the same arguments can be compared output for output.  Compare
with a tolerance: the step is not bit-reproducible from run to run, and two runs of the default command on one B200 (1000 W power
limit) differed by up to 4e-4 of an array's largest magnitude after the 55 training steps, the loss by 6e-7 relative.

``--impl reference`` times the reference's own CPU implementation of the same step on the host cores: the UNMODIFIED
reference modules staged under oracle/_ref by oracle/make_ref.py (h36m.mlp_mixer.MlpMixer / h36m.conv_mixer_model.ConvMixer +
mpjpe_error + torch.optim.Adam, ``kind: "reference"``), on the FULL per-GPU batch, all threads, same config / metric; if
oracle/_ref is not staged it falls back to the torch-CPU port in oracle/mixer_torch.py (``kind: "port"``).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # SURVEY.md §8d K2 / BASELINE.json configs[1]
    "k2": dict(name="MotionMixer MlpMixer+SE, H36M xyz 10->10 frames (22 joints x 3), batch 4096 per GPU",
               family="mlp", B=4096, scale="h36m", loss_scale=1.0,
               cfg=dict(num_classes=66, num_blocks=4, hidden_dim=50, tokens_mlp_dim=20, channels_mlp_dim=50, seq_len=10,
                        pred_len=10, activation="mish", regularization=0.1, input_size=66, r_se=8, use_se=True)),
    # SURVEY.md §8d K1 / BASELINE.json configs[0]: ConvMixer __main__ config (harmonic encoder 64), batch 256
    "k1": dict(name="ConvMixer (train_mixer_h36m.py __main__ config), H36M xyz 10->25 frames (22 joints x 3), batch 256 per GPU",
               family="conv", B=256, scale="h36m", loss_scale=1.0,
               cfg=dict(num_blocks=4, dimPosIn=66, dimPosEmb=50, dimPosOut=66, in_nTP=10, out_nTP=25, conv_nChan=1,
                        conv1_kernel_shape=(1, 3), conv1_stride=(1, 1), conv1_padding=(0, 1), mode_conv="twice", activation="mish",
                        regularization=0.1, use_se=True, r_se=8)),
    # the same ConvMixer at the K2 batch size (large-batch sweep, BASELINE.json configs[4])
    "k1_b4096": dict(name="ConvMixer (train_mixer_h36m.py __main__ config), H36M xyz 10->25 frames, batch 4096 per GPU",
                     family="conv", B=4096, scale="h36m", loss_scale=1.0,
                     cfg=dict(num_blocks=4, dimPosIn=66, dimPosEmb=50, dimPosOut=66, in_nTP=10, out_nTP=25, conv_nChan=1,
                              conv1_kernel_shape=(1, 3), conv1_stride=(1, 1), conv1_padding=(0, 1), mode_conv="twice", activation="mish",
                              regularization=0.1, use_se=True, r_se=8)),
    # SURVEY.md §8d K3 / BASELINE.json configs[2]: ConvMixer AIS autoregressive config (BatchNorm, C=4, E=192, 5x9 / 9x5
    # kernels, 6 blocks), ONE 10 -> 5 pass of the rollout, batch 256
    "k3": dict(name="ConvMixer AIS autoregressive config (BatchNorm, C=4, E=192, k=(5,9)), 10->5 frames (11 joints x 3), batch 256 per GPU",
               family="conv", B=256, scale="ais", loss_scale=1.0,
               cfg=dict(num_blocks=6, dimPosIn=33, dimPosEmb=192, dimPosOut=33, in_nTP=10, out_nTP=5, conv_nChan=4,
                        conv1_kernel_shape=(5, 9), mode_conv="twice", activation="mish", regularization=-1.0, use_se=True, r_se=8,
                        encoder_n_harmonic_functions=0, encoder_omega0=0)),
    # SURVEY.md §8d K4 / BASELINE.json configs[3] (AMASS-shaped), per-GPU batch 4096
    "k4": dict(name="MotionMixer MlpMixer+SE, AMASS-shaped 18 joints 10->25 frames, batch 4096 per GPU",
               family="mlp", B=4096, scale="amass", loss_scale=1000.0,
               cfg=dict(num_classes=54, num_blocks=5, hidden_dim=128, tokens_mlp_dim=20, channels_mlp_dim=128, seq_len=10,
                        pred_len=25, activation="gelu", regularization=0.1, input_size=54, r_se=8, use_se=True)),
}


# stdout carries exactly ONE line (the JSON result): file descriptor 1 is pointed at stderr for the whole run, so that banners
# printed by native libraries (NCCL's "NCCL version ..." when NCCL_DEBUG is set, ...) cannot precede it
_REAL_STDOUT = None


def claim_stdout():
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(obj):
    line = (json.dumps(obj) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(line.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, line)


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 20 ms.  The sampler is started before the warm-up (nvidia-smi takes
    a few hundred ms to produce its first line: longer than a short timed region) and `mark()` brackets the timed region;
    `stop()` reports the samples that fall inside the marks (all samples, and says so, if none did)."""

    Q = ("timestamp,clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc, self.marks = index, [], None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def mark(self):
        self.marks.append(time.time())

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.1)
        self.proc.terminate()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        lo, hi = (self.marks[0], self.marks[-1] + 0.03) if len(self.marks) >= 2 else (0.0, float("inf"))

        def collect(rows):
            sm, mx, reasons = [], [], set()
            for _, r in rows:
                try:
                    sm.append(float(r[1]))
                    mx.append(float(r[2]))
                except (ValueError, IndexError):
                    continue
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            return sorted(sm), mx, reasons

        inside = [row for row in self.rows if lo <= row[0] <= hi]
        sm, mx, reasons = collect(inside)
        window = "timed region"
        if not sm:
            sm, mx, reasons = collect(self.rows)
            window = "warm-up + timed region (no sample fell inside the timed region)"
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "window": window, "reasons": sorted(reasons)}


def common_config(w, world):
    """The `config` object of the JSON line: identical in both arms (ours / reference)."""
    return {"workload": w["name"], "model": {k: (list(v) if isinstance(v, tuple) else v) for k, v in w["cfg"].items()},
            "per_gpu_batch": w["B"], "global_batch": w["B"] * world, "parallelism": "dp%d" % world,
            "optimizer": "Adam lr 1e-3 weight_decay 1e-5", "loss": "MPJPE x %g" % w["loss_scale"]}


class ReferenceTrainer:
    """zero_grad -> model(x) -> mpjpe_error -> backward -> Adam.step with the reference's own modules (oracle/_ref) on the CPU:
    the loop body of h36m/train_mixer_h36m.py:126-193."""

    kind = "reference"

    def __init__(self, w, params):
        import torch
        from oracle.make_ref import import_reference
        MlpMixer, ConvMixer, mpjpe_error = import_reference()
        torch.manual_seed(0)
        self.model = (MlpMixer if w["family"] == "mlp" else ConvMixer)(**w["cfg"])
        if params is not None:
            self.model.load_state_dict(params, strict=True)
        self.model.train()
        self.loss_fn, self.scale = mpjpe_error, w["loss_scale"]
        self.opt = torch.optim.Adam(self.model.parameters(), lr=1e-3, weight_decay=1e-05)

    def step(self, x, gt):
        self.opt.zero_grad()
        loss = self.loss_fn(self.model(x), gt) * self.scale
        loss.backward()
        self.opt.step()
        return loss


def cpu_trainer(w):
    """-> (trainer, kind, description): the real reference when oracle/_ref is staged, else the torch port."""
    import torch
    from oracle import make_ref
    from oracle import mixer_torch as MT
    params = MT.random_params(w["family"], w["cfg"], 0)
    if make_ref.available():
        return ReferenceTrainer(w, None), "reference", "unmodified reference modules (oracle/_ref) + mpjpe_error + torch.optim.Adam, torch %s CPU" % torch.__version__
    return (MT.CpuTrainer(w["family"], w["cfg"], params, loss_scale=w["loss_scale"]), "port",
            "oracle/mixer_torch.py (torch CPU port; oracle/_ref not staged), torch %s" % torch.__version__)


def make_data(w, n_batches, seed):
    from tests.synthetic import synthetic_pose_windows
    c = w["cfg"]
    T, To, D = (c["seq_len"], c["pred_len"], c["input_size"]) if w["family"] == "mlp" else (c["in_nTP"], c["out_nTP"], c["dimPosIn"])
    return [synthetic_pose_windows(w["B"], T, To, D, scale=w["scale"], seed=seed + i) for i in range(n_batches)]


# ---------------------------------------------------------------------------------------------------
def run_reference(args, w):
    """CPU arm (rank 0 only): the reference's own step on the host cores, full per-GPU batch."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    import torch
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    Bs = int(os.environ.get("MMX_CPU_SAMPLE_B", w["B"]))
    wl = dict(w, B=Bs)
    data = [(torch.from_numpy(x), torch.from_numpy(g)) for x, g in make_data(wl, 2, 1234)]
    tr, kind, what = cpu_trainer(w)
    for i in range(args.warmup):
        tr.step(*data[i % 2])
    t0 = time.perf_counter()
    for i in range(args.steps):
        tr.step(*data[i % 2])
    dt = time.perf_counter() - t0
    val = Bs * args.steps / dt
    sample = "%d steps of the %s%d-sequence batch, fp32, %s, %d threads" % (args.steps, "" if Bs == w["B"] else "%d-sequence slice of the " % Bs,
                                                                         w["B"], what, cores)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    emit({
        "impl": "reference", "metric": "train sequences/sec", "value": val, "unit": "sequences/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": common_config(w, world),
        "cpu_baseline": {"value": val, "unit": "sequences/s", "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": val, "unit": "sequences/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    })


def cpu_baseline(w, budget_s=15.0):
    import torch
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    data = [(torch.from_numpy(x), torch.from_numpy(g)) for x, g in make_data(w, 2, 1234)]
    tr, kind, what = cpu_trainer(w)
    tr.step(*data[0])
    n, t0 = 0, time.perf_counter()
    while n < 3 or (time.perf_counter() - t0 < budget_s and n < 40):
        tr.step(*data[n % 2])
        n += 1
    dt = time.perf_counter() - t0
    return {"value": w["B"] * n / dt, "unit": "sequences/s", "cores": cores, "kind": kind,
            "sample": "%d steps of the full %d-sequence batch (%s, fp32, %d threads)" % (n, w["B"], what, cores)}


DUMP_LIMIT = 64 * 2 ** 20


def step_outputs(ts, loss):
    """Host copies of what the last TrainStep.step call computed: the loss it returned, the prediction of its forward pass, the
    parameter gradients and the model's state_dict after its Adam update."""
    import numpy as np
    out = {"loss": np.asarray(loss, dtype=np.float32), "pred": ts.plan.pred.cpu().numpy()}
    for name, off, n, shape in ts._named_flat():
        out["grad." + name] = ts.flat.g[off:off + n].view(shape).cpu().numpy()
    for name, v in ts.model.state_dict().items():
        out["state." + name] = v.cpu().numpy()
    return out


def dump_outputs(path, outputs):
    """DIR/<name>.npy per output, float32 as computed (integer buffers as float64).  If the whole would pass DUMP_LIMIT, the
    prediction is cut to every k-th sequence, the same rows in every run."""
    import numpy as np
    outputs = {k: (v if v.dtype in (np.float32, np.float64) else v.astype(np.float64)) for k, v in outputs.items()}
    rest = sum(v.nbytes for k, v in outputs.items() if k != "pred")
    stride = -(-outputs["pred"].nbytes // max(DUMP_LIMIT - rest, 1))
    outputs["pred"] = outputs["pred"][::stride]
    os.makedirs(path, exist_ok=True)
    for k, v in outputs.items():
        np.save(os.path.join(path, k + ".npy"), v)
    print("bench: %d outputs of the last timed step written to %s (prediction row stride %d)" % (len(outputs), path, stride),
          file=sys.stderr)


# ---------------------------------------------------------------------------------------------------
def run_ours(args, w):
    import torch
    import torch.distributed as dist
    import __graft_entry__ as ge
    ge.build()
    from motionmixerconv_b200 import _lib as L
    from motionmixerconv_b200 import functional as F_
    from motionmixerconv_b200.conv_mixer_model import ConvMixer
    from motionmixerconv_b200.mlp_mixer import MlpMixer
    from motionmixerconv_b200.train import TrainStep

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    pg = None
    if world > 1:
        # rank 0 prints ONE JSON line on stdout: NCCL's own banner ("NCCL version ...", printed when NCCL_DEBUG is set) goes to stderr
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=dev)
        pg = dist.group.WORLD
    torch.manual_seed(0)          # same-seed default initialisation == the reference modules' (sub-modules are built in its order)
    model = MlpMixer(**w["cfg"]) if w["family"] == "mlp" else ConvMixer(**w["cfg"])
    model = model.to(dev).train()
    prec = args.precision if w["family"] == "mlp" else "fp32"      # the tensor-core MixerBlock kernels serve the MlpMixer path
    if w["family"] == "mlp":
        model.set_precision(prec)
    B = w["B"]
    n_batches = 4
    host = [(torch.from_numpy(x).pin_memory(), torch.from_numpy(g).pin_memory()) for x, g in make_data(w, n_batches, 1234 + 1000 * rank)]
    devd = [(x.to(dev), g.to(dev)) for x, g in host]
    ts = TrainStep(model, lr=1e-3, weight_decay=1e-5, loss_scale=w["loss_scale"], process_group=pg)
    flush = torch.empty(512 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)   # 512 MB > 126 MB L2

    loss_pinned = [torch.zeros((), dtype=torch.float32).pin_memory() for _ in range(2)]
    loss_ready = [torch.cuda.Event() for _ in range(2)]

    def timed(n_steps, data, read_loss, ts=ts, sync_read=False):
        """read_loss: the end-to-end arm (host inputs, loss read back every step).  sync_read=False: the loss of step i is copied
        to pinned host memory asynchronously and consumed by the host while step i+1 runs (what a training loop that logs
        its loss does; the reference's loop only accumulates it on the device, train_mixer_h36m.py:195); sync_read=True: the
        host blocks on every step's loss before launching the next step."""
        evs, seen = [], []
        for i in range(n_steps):
            flush.add_(1.0)                       # evict L2 between timed iterations (outside the events)
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            if read_loss:      # end-to-end arm: this step's host inputs were prefetched during the previous step; prefetch the next
                loss = ts.step(*data[i % n_batches], prefetch=data[(i + 1) % n_batches])
            else:
                loss = ts.step(*data[i % n_batches])
            if read_loss and sync_read:
                seen.append(float(loss.to("cpu", non_blocking=False)))   # D2H read of the step's result, host blocks
            elif read_loss:
                loss_pinned[i % 2].copy_(loss, non_blocking=True)        # D2H read of the step's result inside the region
                loss_ready[i % 2].record()
                if i > 0:                                                # the host consumes the previous step's loss
                    loss_ready[(i - 1) % 2].synchronize()
                    seen.append(float(loss_pinned[(i - 1) % 2]))
            e.record()
            evs.append((s, e))
        torch.cuda.synchronize(dev)
        if read_loss and not sync_read:
            seen.append(float(loss_pinned[(n_steps - 1) % 2]))
        assert not read_loss or len(seen) == n_steps
        per_step = sorted(s.elapsed_time(e) for s, e in evs)
        timed.median_ms = per_step[len(per_step) // 2]
        return sum(per_step), float(loss)

    def barrier():
        if world > 1:
            dist.barrier(device_ids=[local])
        torch.cuda.synchronize(dev)

    # ---- device-resident arm (value) ----
    sampler = ClockSampler(local)
    sampler.start()
    timed(args.warmup, devd, False)
    barrier()
    sampler.mark()
    t_ms, last_loss = timed(args.steps, devd, False)
    median_ms = timed.median_ms
    barrier()
    # copied now: the arms below train the same model further
    outputs = step_outputs(ts, last_loss) if args.dump_outputs and rank == 0 else None
    # ---- data parallel: every rank must hold bit-identical parameters after the timed steps
    dp_identical = None
    if world > 1:
        pmax, pmin = ts.flat.p.clone(), ts.flat.p.clone()
        dist.all_reduce(pmax, op=dist.ReduceOp.MAX)
        dist.all_reduce(pmin, op=dist.ReduceOp.MIN)
        dp_identical = bool(torch.equal(pmax, pmin))
    # ---- end-to-end arm: pinned host inputs, H2D inside the region, loss read back every step ----
    timed(max(1, args.warmup // 2), host, True)
    barrier()
    t_e2e_ms, _ = timed(args.steps, host, True)
    barrier()
    timed(1, host, True, sync_read=True)
    barrier()
    t_e2e_sync_ms, _ = timed(args.steps, host, True, sync_read=True)
    barrier()
    sampler.mark()
    clocks = sampler.stop()
    # ---- the other arithmetic mode of the same step (device-resident), for the record ----
    t_alt_ms, alt = 0.0, None
    if w["family"] == "mlp" and not args.no_alt_precision:
        alt = "fp32" if prec == "tf32" else "tf32"
        torch.manual_seed(0)
        model2 = MlpMixer(**w["cfg"]).to(dev).train().set_precision(alt)
        ts2 = TrainStep(model2, lr=1e-3, weight_decay=1e-5, loss_scale=w["loss_scale"], process_group=pg)
        timed(args.warmup, devd, False, ts2)
        barrier()
        t_alt_ms, _ = timed(args.steps, devd, False, ts2)
        barrier()
    tt = torch.tensor([t_ms, t_e2e_ms, t_alt_ms, t_e2e_sync_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    t_ms, t_e2e_ms, t_alt_ms, t_e2e_sync_ms = tt.tolist()

    # ---- dominant kernel timed alone for the roofline ----
    roof = None
    if rank == 0:
        import ctypes as C
        lib = L.load()
        pl = ts.plan
        st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        c = w["cfg"]
        peak, which = peaks()
        fp32_peak = 148 * 128 * 2 * 1.965e9 / 1e12     # fp32 FMA pipe: 148 SMs x 128 lanes x 2 flop x 1.965 GHz (nominal)

        def time_kernel(call, reps=20):
            tot = 0.0
            for i in range(reps + 3):
                flush.add_(1.0)
                s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                s.record()
                call()
                e.record()
                torch.cuda.synchronize(dev)
                if i >= 3:
                    tot += s.elapsed_time(e)
            return tot / reps

        others = {}
        if w["family"] == "mlp":
            mb, tw, tg = pl.blocks[1]
            d = pl._desc(mb, True)
            tile = c["seq_len"] * c["hidden_dim"] * 4
            T_, H_, tok_, ch_ = c["seq_len"], c["hidden_dim"], c["tokens_mlp_dim"], c["channels_mlp_dim"]
            if pl.saves[1]:
                # tcgen05 family: the block backward is two kernels; the dominant one is the channel half (tensor cores)
                x1, gate = pl.x1[1], pl.gate[1]
                t_ch = time_kernel(lambda: L.check(lib, lib.mmx_mlp_channel_half_bwd(C.byref(d), C.byref(tw), C.byref(tg), x1.data_ptr(),
                                                                                     pl.dact[0].data_ptr(), pl.dact[1].data_ptr(), st), "channel_half_bwd"))
                t_tk = time_kernel(lambda: L.check(lib, lib.mmx_mlp_token_half_bwd(C.byref(d), C.byref(tw), C.byref(tg), pl.acts[1].data_ptr(),
                                                                                   x1.data_ptr(), gate.data_ptr(), pl.dact[1].data_ptr(),
                                                                                   pl.dact[1].data_ptr(), st), "token_half_bwd"))
                t_cf = time_kernel(lambda: L.check(lib, lib.mmx_mlp_channel_half_fwd(C.byref(d), C.byref(tw), x1.data_ptr(), pl.acts[2].data_ptr(), st), "channel_half_fwd"))
                t_tf = time_kernel(lambda: L.check(lib, lib.mmx_mlp_token_half_fwd(C.byref(d), C.byref(tw), pl.acts[1].data_ptr(), x1.data_ptr(),
                                                                                   gate.data_ptr(), st), "token_half_fwd"))
                others = {"token_half_bwd_ms": t_tk, "channel_half_fwd_ms": t_cf, "token_half_fwd_ms": t_tf,
                          "block_fwd_bwd_GBps": B * 9 * tile / ((t_ch + t_tk + t_cf + t_tf) * 1e-3) / 1e9,
                          "block_fwd_bwd_frac": B * 9 * tile / ((t_ch + t_tk + t_cf + t_tf) * 1e-3) / 1e9 / peak,
                          "block_bytes_note": "save variant, per sequence: fwd token x->x1 (2 tiles) + channel x1->y (2); bwd channel x1,dy->dx1 (3) "
                                              "+ token x,x1,dx1->dx (4) = 11 tile transfers, 9 algorithmic (x1 written once, dx1 in place)"}
                t_k = t_ch
                kname = "chan_bwd_kernel (MixerBlock channel half backward: tcgen05.mma bf16x3, accumulators + dW in TMEM, UBLKCP tiles)"
                # six contractions [rows,H]x[H,ch] (fwd recompute 2, data gradients 2, weight gradients 2), 3 MMAs each
                flops = B * 6 * 2 * T_ * H_ * ch_
                tensor_flops = 3 * flops
            else:
                t_k = time_kernel(lambda: L.check(lib, lib.mmx_mlp_block_bwd(C.byref(d), C.byref(tw), C.byref(tg), pl.acts[1].data_ptr(),
                                                                             pl.dact[0].data_ptr(), pl.dact[1].data_ptr(), st), "mmx_mlp_block_bwd"))
                kname = "mlp_block_bwd (MixerBlock backward, forward recomputed in-kernel)"
                flops = B * 4 * 2 * T_ * (2 * tok_ * H_ + 2 * H_ * ch_)
                tensor_flops = None
        else:
            kind, mb, half, tw, tg = pl.ops[2]
            d = pl._desc(mb, half, True)
            if 2 in pl.bn:          # BatchNorm half: time the second backward pass (BN + conv + LN backward)
                b = pl.bn[2]
                coef = torch.zeros(3 * c["conv_nChan"], device=dev)
                call = lambda: L.check(lib, lib.mmx_conv_half_bn_bwd2(C.byref(d), C.byref(tw), C.byref(tg), b["bn"].data_ptr(), coef.data_ptr(),
                                                                      pl.acts[2].data_ptr(), b["z"].data_ptr(), pl.dact[0].data_ptr(),
                                                                      b["gd"].data_ptr(), pl.dact[1].data_ptr(), st), "mmx_conv_half_bn_bwd2")
            else:
                call = lambda: L.check(lib, lib.mmx_conv_half_bwd(C.byref(d), C.byref(tw), C.byref(tg), pl.acts[2].data_ptr(), pl.dact[0].data_ptr(),
                                                                  pl.dact[1].data_ptr(), st), "mmx_conv_half_bwd")
            t_k = time_kernel(call)
            tile = c["conv_nChan"] * c["in_nTP"] * c["dimPosEmb"] * 4
            kname = "conv_half_bwd (one ConvMixerBlock half backward, forward recomputed in-kernel)"
            kt, kp = mb.conv1.kernel
            flops = B * 4 * 2 * c["conv_nChan"] ** 2 * kt * kp * c["in_nTP"] * c["dimPosEmb"]
            tensor_flops = None
        alg = B * 3 * tile                      # read block-half input + upstream grad, write input grad
        ach = alg / (t_k * 1e-3) / 1e9
        traffic, traffic_src = None, None
        tpath = os.path.join(ROOT, "profiles", "roofline_traffic.json")
        if os.path.exists(tpath):
            with open(tpath) as f:
                tj = json.load(f)
                ent = tj.get(args.workload + "_" + prec) or tj.get(args.workload)
            if ent:
                traffic, traffic_src = ent["bytes"], ent["source"]
        roof = {"kernel": kname, "bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                "peak_source": which, "algorithmic_bytes_per_launch": alg, "kernel_ms": t_k, "traffic": traffic,
                "traffic_source": traffic_src,
                "math_tflops": flops / (t_k * 1e-3) / 1e12, "fp32_pipe_frac_if_simt": flops / (t_k * 1e-3) / 1e12 / fp32_peak,
                "note": ("tcgen05 family: the kernel is bound by instruction issue / latency of the fp32 epilogue work between the MMAs "
                         "(LayerNorm, activation, dropout, operand split, SE) and by the per-CTA prologue at 2-3 tiles per CTA, not by "
                         "HBM or the tensor pipe" if tensor_flops else
                         "fp32 SIMT (1e-5 parity mode): the kernel is bound by the fp32 pipe / latency, not HBM") + " — see DESIGN.md §4"}
        if tensor_flops:
            roof["tensor_tflops_issued"] = tensor_flops / (t_k * 1e-3) / 1e12
        roof.update(others)

    def shutdown():
        """Tear the process group down without ever blocking the benchmark's exit (the JSON line is already out)."""
        if world <= 1:
            return
        ts.release_graphs()
        if alt:
            ts2.release_graphs()
        killer = threading.Timer(20.0, lambda: os._exit(0))
        killer.daemon = True
        killer.start()
        dist.destroy_process_group()
        killer.cancel()

    if rank != 0:
        shutdown()
        return
    c = w["cfg"]
    x0, g0 = host[0]
    tc5 = w["family"] == "mlp" and prec == "tf32" and any(ts.plan.saves)
    out = {
        "metric": "train sequences/sec", "value": world * B * args.steps / (t_ms * 1e-3), "unit": "sequences/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": t_ms / args.steps,
        "ms_per_step_median": median_ms,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16x3 (MixerBlock channel-MLP contractions: bf16 hi+lo split operands, fp32 accumulate in TMEM); everything else f32" if tc5 else "f32",
        "data": "synthetic",
        "config": common_config(w, world),
        "details": {
            "precision": ("reduced-precision mode of the north star (2e-3 bar; measured 5e-6..3e-5 vs the fp64 oracle): tcgen05 kernel family -- "
                          "channel MLP on the tensor cores (bf16 split operands, 3 MMAs per product), token MLP on packed-fp32 CUDA cores; LayerNorm, "
                          "activations, SE, residuals, loss, Adam and the embed / head kernels fp32") if tc5 else
                         ("fp32 everywhere (north star: 1e-5 parity mode)" if prec == "fp32" else "tf32 requested; shape served by the fp32 kernels"),
            "l2": "512 MB L2 flush between timed iterations (outside the CUDA-event pairs)",
            "step": "CUDA graph A: memset + embed/encoder + block kernels fwd + head + mpjpe + head bwd + block kernels bwd + embed/encoder bwd"
                    + ("; fused Adam" if world == 1 else
                       ("; ONE kernel: all-reduce of the flat gradient bucket over NVLink peer memory + Adam (mmx_adam_step_peer), the whole step is one graph"
                        if ts.peer is not None else "; NCCL all-reduce of the flat gradient bucket; fused Adam (graph B)")),
            "timing": "CUDA events around every step on the launching stream; value = B x steps / sum of the K step times (max over ranks); "
                      "ms_per_step_median = median of the K per-step times"},
        "e2e": {"value": world * B * args.steps / (t_e2e_ms * 1e-3), "unit": "sequences/s",
                "h2d_bytes_per_step": x0.numel() * 4 + g0.numel() * 4, "d2h_bytes_per_step": 4,
                "ms_per_step": t_e2e_ms / args.steps,
                "host_sync_every_step": {"value": world * B * args.steps / (t_e2e_sync_ms * 1e-3), "unit": "sequences/s",
                                         "ms_per_step": t_e2e_sync_ms / args.steps,
                                         "note": "the same loop with loss.to('cpu') blocking the host before the next step is launched"},
                "note": "TrainStep.step(x_host, gt_host, prefetch=next): every step's inputs cross PCIe from pinned memory inside the "
                        "timed region (double-buffered on a copy stream, overlapping the previous step's kernels); every step's loss is "
                        "copied to pinned host memory inside the region and read by the host while the next step runs (one step of lag, "
                        "as a loop that logs its loss; the reference's loop only accumulates it on the device, train_mixer_h36m.py:195)"},
        "gpu_launches": ts.kernel_launches_per_step * args.steps,
        "final_loss": last_loss,
        "clocks": clocks,
        "roofline": roof,
    }
    if dp_identical is not None:
        out["dp_params_identical"] = dp_identical
    if alt:
        out["other_precision"] = {"precision": alt, "value": world * B * args.steps / (t_alt_ms * 1e-3), "unit": "sequences/s",
                                  "ms_per_step": t_alt_ms / args.steps}
    if world == 1 and not args.no_cpu_baseline:
        out["cpu_baseline"] = cpu_baseline(w)
    if outputs is not None:
        dump_outputs(args.dump_outputs, outputs)
    emit(out)
    shutdown()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=os.environ.get("MMX_WORKLOAD", "k2"), choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--precision", default=os.environ.get("MMX_BENCH_PRECISION", "tf32"), choices=["fp32", "tf32"],
                    help="arithmetic of the MixerBlock contractions: tf32 = the north star's reduced-precision (2e-3) mode, served by the "
                         "tcgen05 kernel family (default, the headline); fp32 = the 1e-5 mode on fp32 SIMT kernels")
    ap.add_argument("--no-alt-precision", action="store_true", help="skip the extra timing of the other precision mode")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed (loss, prediction, gradients, "
                    "state_dict after the update) as DIR/<name>.npy, at most 64 MB in all")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    claim_stdout()
    args.warmup = max(args.warmup, 3)
    w = WORKLOADS[args.workload]
    if args.impl == "reference":
        run_reference(args, w)
    else:
        run_ours(args, w)


if __name__ == "__main__":
    main()
