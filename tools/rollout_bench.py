"""BASELINE.json configs[2]: ConvMixer AIS-shaped autoregressive rollout (25-frame prediction = 5 chained 10 -> 5 passes),
training (BPTT through the predictions + Adam, RolloutTrainer graph) and inference (RolloutExecutor graph), at the
reference's batch size 50 and at 256 / 4096, next to the eager path and the reference's CPU step (reference modules from
oracle/_ref driven by the same loop on the host cores).  One JSON line per cell.  Under torchrun (N GPUs): every rank rolls out its
own batch of B sequences (weak scaling), the training step exchanges gradients inside the fused optimiser; values are whole-job
(N x B / max-over-ranks time); the eager and CPU cells are skipped."""
import json
import os
import sys
import time
from argparse import Namespace

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from motionmixerconv_b200.conv_mixer_model import ConvMixer
from motionmixerconv_b200.rollout import RolloutExecutor, RolloutTrainer, autoregressive_process_batch
from motionmixerconv_b200.train import FusedAdam
from tests.synthetic import synthetic_full_windows

RANK, WORLD, LOCAL = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0))
torch.cuda.set_device(LOCAL)
PG = None
if WORLD > 1:
    import torch.distributed as dist
    dist.init_process_group("nccl", device_id=torch.device("cuda", LOCAL))
    PG = dist.group.WORLD

CFG = dict(num_blocks=6, dimPosIn=33, dimPosEmb=192, dimPosOut=33, in_nTP=10, out_nTP=5, conv_nChan=4, conv1_kernel_shape=(5, 9),
           mode_conv="twice", activation="mish", regularization=-1.0, use_se=True, r_se=8, encoder_n_harmonic_functions=0, encoder_omega0=0)
ARGS = Namespace(input_n_dataset=10, output_n_dataset=25, input_n_model=10, output_n_model=5, step_window=5, loss_type="mpjpe")
DIM = list(range(33))


def timed(fn, n, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(n):
        fn()
    e.record()
    torch.cuda.synchronize()
    ms = s.elapsed_time(e) / n
    if WORLD > 1:
        t = torch.tensor([ms], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t)
    return ms


def cpu_cell(B, train):
    from oracle import make_ref
    if not make_ref.available():
        return None
    _, Conv, mpjpe = make_ref.import_reference()
    torch.set_num_threads(os.cpu_count() or 1)
    torch.manual_seed(0)
    m = Conv(**CFG)
    batch = torch.from_numpy(synthetic_full_windows(B, 35, 33, scale="ais", seed=1))
    if train:
        m.train()
        opt = torch.optim.Adam(m.parameters(), lr=1e-3, weight_decay=1e-5)

        def step():
            opt.zero_grad()
            loss, _ = autoregressive_process_batch(batch, m, ARGS, DIM, False, loss_fn=mpjpe)
            loss.backward()
            opt.step()
    else:
        m.eval()

        def step():
            with torch.no_grad():
                autoregressive_process_batch(batch, m, ARGS, DIM, False, loss_fn=mpjpe)
    step()
    n, t0 = 0, time.perf_counter()
    while n < 2 or (time.perf_counter() - t0 < 6 and n < 20):
        step()
        n += 1
    dt = (time.perf_counter() - t0) / n
    return {"value": B / dt, "unit": "sequences/s", "ms": dt * 1e3, "cores": os.cpu_count(), "kind": "reference modules (oracle/_ref) + the rollout loop",
            "sample": "%d rollouts of %d sequences" % (n, B)}


for B in [int(v) for v in os.environ.get("ROLLOUT_B", "50,256,4096").split(",")]:
    torch.manual_seed(0)
    batch = torch.from_numpy(synthetic_full_windows(B, 35, 33, scale="ais", seed=1 + RANK)).cuda()
    cell = {"workload": "ConvMixer AIS autoregressive rollout (K3: BatchNorm, C=4, E=192, k=(5,9), 6 blocks), 10 -> 25 frames as 5 chained passes",
            "per_gpu_batch": B, "n_gpus": WORLD}
    # training, graph
    model = ConvMixer(**CFG).cuda().train()
    tr = RolloutTrainer(model, ARGS, DIM, teacher_forcing=False, process_group=PG)
    ms = timed(lambda: tr.step(batch), 10)
    cell["train_graph"] = {"ms": ms, "value": WORLD * B / ms * 1e3, "unit": "sequences/s", "nan": bool(tr.nan_flag)}
    if WORLD > 1:
        pmax, pmin = tr.opt.flat(0).p.clone(), tr.opt.flat(0).p.clone()
        dist.all_reduce(pmax, op=dist.ReduceOp.MAX)
        dist.all_reduce(pmin, op=dist.ReduceOp.MIN)
        cell["dp_params_identical"] = bool(torch.equal(pmax, pmin))
        ex = RolloutExecutor(model.eval(), 10, 25, 10, 5, 5)
        ms = timed(lambda: ex(batch), 20)
        cell["infer_graph"] = {"ms": ms, "value": WORLD * B / ms * 1e3, "unit": "sequences/s"}
        if RANK == 0:
            print(json.dumps(cell), flush=True)
        del model, tr, ex
        torch.cuda.empty_cache()
        continue
    # training, eager autograd (what round 1 had)
    model2 = ConvMixer(**CFG).cuda().train()
    opt = FusedAdam(model2.parameters(), lr=1e-3, weight_decay=1e-5)

    def eager():
        opt.zero_grad(set_to_none=True)
        loss, _ = autoregressive_process_batch(batch, model2, ARGS, DIM, False)
        loss.backward()
        opt.step()
    ms = timed(eager, 5)
    cell["train_eager"] = {"ms": ms, "value": B / ms * 1e3, "unit": "sequences/s"}
    # inference, graph
    ex = RolloutExecutor(model.eval(), 10, 25, 10, 5, 5)
    ms = timed(lambda: ex(batch), 20)
    cell["infer_graph"] = {"ms": ms, "value": B / ms * 1e3, "unit": "sequences/s"}
    if os.environ.get("ROLLOUT_CPU", "1") == "1" and B <= 256:
        cell["cpu_train"] = cpu_cell(B, True)
        cell["cpu_infer"] = cpu_cell(B, False)
    print(json.dumps(cell), flush=True)
    del model, model2, tr, ex, opt
    torch.cuda.empty_cache()

if WORLD > 1:
    import threading
    threading.Timer(15.0, lambda: os._exit(0)).start()
    dist.destroy_process_group()
    os._exit(0)
