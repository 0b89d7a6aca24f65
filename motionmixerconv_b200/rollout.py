"""Autoregressive sliding-window rollout — drop-in for ``autoregressive_process_batch``
(``h36m/train_autoreg_mixer_h36m.py:195-258``, called from ``train_autoreg_mixer_ais.py:151-153``).

Training keeps the reference semantics exactly: chained ``model(subsequence)`` calls, the loss summed over the windows and
divided by ``output_n_dataset // step_window``, gradients flowing through the predictions when ``teacher_forcing`` is off
(no detach, ``:243-253``).  Every forward / backward is the fused sm_100a kernels via the autograd Functions.

``RolloutExecutor`` is the inference fast path (``test_mpjpe_autoregressive``, ``:261-357``): the whole chain of forward
passes, the window shifts and the writes into ``full_sequence_predict`` are captured once in a CUDA graph and replayed per
batch; there is no per-window Python, no per-batch ``isnan`` host sync (the reference's ``:256``).
"""
from __future__ import annotations

import torch

from .functional import angle_l1_error, mpjpe_error


def _windows(args):
    return range(0, args.input_n_dataset + args.output_n_dataset - args.input_n_model - args.output_n_model + 1, args.step_window)


def autoregressive_process_batch(batch, model, args, dim_used, teacher_forcing, check_nan=False, loss_fn=None):
    """Same signature / return as the reference: ``(loss / n_windows, full_sequence_predict)``.

    ``check_nan=True`` restores the reference's ``assert not torch.isnan(loss)`` (``:256``), which costs a host
    synchronisation per batch; the default leaves the check to the caller (``RolloutTrainer.nan_flag`` keeps it on the
    device).  ``loss_fn``: override of the MPJPE loss (used by the CPU baseline, which runs this loop over the reference's
    own modules)."""
    assert args.output_n_dataset % args.step_window == 0, "output_n_dataset does not divide by step_window"
    assert args.output_n_dataset // args.step_window >= 1, "output_n_dataset is smaller than step_window"
    if loss_fn is not None:
        loss_fct = lambda pred, gt, out_n: loss_fn(pred, gt)
    elif args.loss_type == 'mpjpe':
        loss_fct = lambda pred, gt, out_n: mpjpe_error(pred, gt)
    elif args.loss_type == 'angle':
        loss_fct = lambda pred, gt, out_n: angle_l1_error(pred.reshape(-1, out_n, len(dim_used)), gt)
    else:
        raise ValueError("unknown loss_type %s" % args.loss_type)
    full_sequence = batch[:, :args.input_n_dataset + args.output_n_dataset, dim_used].clone()
    full_sequence_gt = batch[:, args.input_n_dataset:args.input_n_dataset + args.output_n_dataset, dim_used].clone()
    full_sequence_predict = torch.zeros_like(full_sequence_gt)
    subsequence_train = full_sequence[:, 0: args.input_n_model, :]
    loss = torch.zeros(1, device=batch.device)
    for start in _windows(args):
        end_train = start + args.input_n_model
        end_predict = end_train + args.output_n_model
        if teacher_forcing:
            subsequence_train = full_sequence[:, start:end_train, :]
        subsequence_gt = full_sequence[:, end_train:end_predict, :]
        subsequence_predict = model(subsequence_train.contiguous())
        loss = loss + loss_fct(subsequence_predict, subsequence_gt.contiguous(), args.output_n_model)
        full_sequence_predict[:, end_train - args.input_n_model: end_predict - args.input_n_model, :] = subsequence_predict.detach()
        if not teacher_forcing:
            frames_to_take = args.input_n_model - args.step_window
            subsequence_train = torch.cat((subsequence_train[:, -frames_to_take:, :], subsequence_predict), dim=1)
    if check_nan:
        assert not torch.isnan(loss), 'Loss is nan'
    return loss / (args.output_n_dataset // args.step_window), full_sequence_predict


class RolloutExecutor:
    """CUDA-graph inference rollout: ``predict = ex(full_sequence)``.

    ``full_sequence``: [B, input_n_dataset + output_n_dataset, D] (only the first ``input_n_model`` frames are read when
    ``teacher_forcing`` is off, as in evaluation).  Returns [B, output_n_dataset, D_out] — the reference's
    ``full_sequence_predict``.  The model is put in ``eval()`` semantics for the captured passes.
    """

    def __init__(self, model, input_n_dataset, output_n_dataset, input_n_model, output_n_model, step_window, teacher_forcing=False):
        assert output_n_dataset % step_window == 0 and output_n_dataset // step_window >= 1
        if not teacher_forcing and input_n_model - step_window + output_n_model != input_n_model:
            raise ValueError("step_window must equal output_n_model for a free-running rollout (window length stays input_n_model)")
        self.model = model
        self.n_in_ds, self.n_out_ds = input_n_dataset, output_n_dataset
        self.n_in, self.n_out, self.step = input_n_model, output_n_model, step_window
        self.teacher_forcing = teacher_forcing
        self.starts = list(range(0, input_n_dataset + output_n_dataset - input_n_model - output_n_model + 1, step_window))
        self.graph = None
        self.B = None

    def _run(self):
        win = self.seq[:, :self.n_in, :]
        for start in self.starts:
            end_train = start + self.n_in
            if self.teacher_forcing:
                win = self.seq[:, start:end_train, :]
            pred = self.model(win.contiguous())
            self.out[:, start:start + self.n_out, :] = pred
            if not self.teacher_forcing:
                win = torch.cat((win[:, self.step:, :], pred), dim=1)

    @torch.no_grad()
    def __call__(self, full_sequence):
        if not full_sequence.is_cuda:
            raise RuntimeError("RolloutExecutor needs CUDA tensors (the hot path has no CPU implementation)")
        was_training = self.model.training
        self.model.eval()
        try:
            if self.graph is None or self.B != full_sequence.shape[0]:
                self.B = full_sequence.shape[0]
                self.seq = torch.empty_like(full_sequence, memory_format=torch.contiguous_format)
                self.seq.copy_(full_sequence)
                probe = self.model(self.seq[:, :self.n_in, :].contiguous())          # warm-up (kernel attributes) + output width
                self.out = torch.zeros(self.B, self.n_out_ds, probe.shape[-1], device=full_sequence.device)
                side = torch.cuda.Stream()
                side.wait_stream(torch.cuda.current_stream())
                with torch.cuda.stream(side):
                    self._run()
                torch.cuda.current_stream().wait_stream(side)
                self.graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(self.graph):
                    self._run()
            self.seq.copy_(full_sequence)
            self.graph.replay()
            return self.out
        finally:
            self.model.train(was_training)


class RolloutTrainer:
    """One optimisation step of the autoregressive training loop (``train_autoregressive``, train_autoreg_mixer_h36m.py:110-135:
    ``zero_grad; loss, _ = autoregressive_process_batch(...); loss.backward(); optimizer.step()``) as ONE CUDA-graph replay:
    the chained forward passes, the window concatenations, the per-window losses, back-propagation through the predictions
    (no teacher forcing) and the fused Adam update are captured once per batch shape.  The NaN check of the reference stays on
    the device (``nan_flag``), so there is no host synchronisation in the loop.

        tr = RolloutTrainer(model, args, dim_used, teacher_forcing=False, lr=1e-3)
        loss, predict = tr.step(batch)          # static tensors, valid until the next step
    """

    def __init__(self, model, args, dim_used, teacher_forcing=False, lr=1e-3, weight_decay=1e-5, use_cuda_graph=True, process_group=None):
        """``process_group``: batch-sharded data parallelism (every rank rolls out its own shard; the gradient exchange is part
        of the fused optimiser step, see FusedAdam).  BatchNorm statistics stay per replica; model buffers are broadcast from
        rank 0 at construction."""
        from .train import FusedAdam
        self.model, self.args, self.teacher_forcing = model, args, teacher_forcing
        self.dim_used = dim_used          # index tensor on the device is made at the first step (no host->device copy inside the capture)
        self.opt = FusedAdam(model.parameters(), lr=lr, weight_decay=weight_decay, process_group=process_group)
        if process_group is not None:
            import torch.distributed as dist
            for gi in range(len(self.opt.param_groups)):           # flat buffers + rank 0's parameters now (not inside the capture warm-up)
                self.opt.flat(gi)
            for b in model.buffers():
                dist.broadcast(b, src=dist.get_global_rank(process_group, 0), group=process_group)
        self.use_graph = use_cuda_graph
        self.graph = None
        self.batch = None
        self.loss = self.predict = self.nan_flag = None
        self.step_dev = None

    def _body(self):
        from . import functional as F_
        if self.step_dev is None:
            self.step_dev = torch.zeros(1, dtype=torch.int32, device=self.batch.device)
        F_.set_dropout_step_tensor(self.step_dev)      # dropout masks advance with a device-side counter (graph replays)
        try:
            loss, predict = autoregressive_process_batch(self.batch, self.model, self.args, self.dim_used, self.teacher_forcing, check_nan=False)
            loss.backward()
        finally:
            F_.set_dropout_step_tensor(None)
        self.opt.step()
        self.step_dev.add_(len(_windows(self.args)))
        return loss.detach().reshape(()), predict, torch.isnan(loss.detach()).reshape(())

    def step(self, batch):
        if not batch.is_cuda:
            raise RuntimeError("RolloutTrainer needs CUDA tensors (the hot path has no CPU implementation)")
        if not self.model.training:
            raise RuntimeError("RolloutTrainer.step: the model is in eval() mode")
        if not isinstance(self.dim_used, torch.Tensor) or self.dim_used.device != batch.device:
            self.dim_used = torch.as_tensor(list(self.dim_used), dtype=torch.long).to(batch.device)
        if not self.use_graph:
            self.batch = batch
            self.opt.zero_grad(set_to_none=True)
            self.loss, self.predict, self.nan_flag = self._body()
            return self.loss, self.predict
        if self.graph is None or self.batch.shape != batch.shape:
            self.batch = batch.clone()
            side = torch.cuda.Stream(device=batch.device)
            side.wait_stream(torch.cuda.current_stream())
            # whole-step capture (fwd + bwd + optimiser): warm up on a side stream, restore the state the warm-up steps changed
            state = [p.detach().clone() for p in self.model.parameters()] + [b.detach().clone() for b in self.model.buffers()]
            with torch.cuda.stream(side):
                for _ in range(2):
                    self.opt.zero_grad(set_to_none=True)
                    self._body()
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            with torch.no_grad():
                for t, sv in zip(list(self.model.parameters()) + list(self.model.buffers()), state):
                    t.copy_(sv)
                for f in self.opt._flat.values():
                    f.m.zero_(); f.v.zero_(); f.step.zero_()
                self.step_dev.zero_()
            for m in self.model.modules():
                if hasattr(m, "_calls"):
                    m._calls = 0                      # dropout step counters of the blocks
            self.opt.zero_grad(set_to_none=True)
            self.graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph):
                self.loss, self.predict, self.nan_flag = self._body()
            # the capture itself did not execute anything: parameters / optimiser state are those before the first step
        self.batch.copy_(batch)
        self.graph.replay()
        return self.loss, self.predict
