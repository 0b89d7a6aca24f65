"""Drop-in replacement for the reference ``h36m/mlp_mixer.py`` (MotionMixer ``MlpMixer``).

Same constructor arguments (mlp_mixer.py:254-258), same ``forward(x)`` signature, same
``state_dict`` keys / shapes / registration order, same default initialisation from the same
``torch.manual_seed`` (the sub-modules are created in the reference's construction order so the RNG
draws line up).  The sub-modules are *parameter holders*: all arithmetic of ``forward`` runs in the
fused sm_100a kernels behind ``motionmixerconv_b200.functional``.
"""
from __future__ import annotations

import torch
import torch.nn as nn

from . import functional as F_


class SELayer(nn.Module):
    """Parameter holder for the squeeze-excitation over frames (mlp_mixer.py:6-34)."""

    def __init__(self, c, r=4, use_max_pooling=False):
        super().__init__()
        self.squeeze = nn.AdaptiveAvgPool1d(1) if not use_max_pooling else nn.AdaptiveMaxPool1d(1)
        self.excitation = nn.Sequential(
            nn.Linear(c, c // r, bias=False),
            nn.ReLU(inplace=True),
            nn.Linear(c // r, c, bias=False),
            nn.Sigmoid(),
        )
        self.use_max_pooling = use_max_pooling

    def forward(self, x):
        raise NotImplementedError("SELayer is fused into MixerBlock.forward (no standalone kernel)")


class MlpBlock(nn.Module):
    """Parameter holder for fc1 -> act -> reg1 -> fc2 -> reg2 (mlp_mixer.py:44-96)."""

    def __init__(self, mlp_hidden_dim, mlp_input_dim, mlp_bn_dim, activation='gelu', regularization=0, initialization='none'):
        super().__init__()
        self.mlp_hidden_dim = mlp_hidden_dim
        self.mlp_input_dim = mlp_input_dim
        self.mlp_bn_dim = mlp_bn_dim
        self.fc1 = nn.Linear(self.mlp_input_dim, self.mlp_hidden_dim)
        self.fc2 = nn.Linear(self.mlp_hidden_dim, self.mlp_input_dim)
        if regularization > 0.0:
            self.reg1 = nn.Dropout(regularization)
            self.reg2 = nn.Dropout(regularization)
        elif regularization == -1.0:
            self.reg1 = nn.BatchNorm1d(self.mlp_bn_dim)
            self.reg2 = nn.BatchNorm1d(self.mlp_bn_dim)
        else:
            self.reg1 = None
            self.reg2 = None
        if activation not in ('gelu', 'mish'):
            raise ValueError('Unknown activation function type: %s' % activation)
        self.activation = activation

    def forward(self, x):
        raise NotImplementedError("MlpBlock is fused into MixerBlock.forward (no standalone kernel)")


class MixerBlock(nn.Module):
    """One fused kernel forward, one backward (mlp_mixer.py:100-164, functional.FusedMixerBlock); with regularization == -1
    (BatchNorm1d) a chain of stage kernels around the batch reductions (functional.MlpBnBlock)."""

    def __init__(self, tokens_mlp_dim, channels_mlp_dim, seq_len, hidden_dim, activation='gelu', regularization=0,
                 initialization='none', r_se=4, use_max_pooling=False, use_se=True):
        super().__init__()
        self.tokens_mlp_dim = tokens_mlp_dim
        self.channels_mlp_dim = channels_mlp_dim
        self.seq_len = seq_len
        self.hidden_dim = hidden_dim
        self.mlp_block_token_mixing = MlpBlock(self.tokens_mlp_dim, self.seq_len, self.hidden_dim, activation=activation,
                                               regularization=regularization, initialization=initialization)
        self.mlp_block_channel_mixing = MlpBlock(self.channels_mlp_dim, self.hidden_dim, self.seq_len, activation=activation,
                                                 regularization=regularization, initialization=initialization)
        self.use_se = use_se
        if self.use_se:
            self.se = SELayer(self.seq_len, r=r_se, use_max_pooling=use_max_pooling)
        self.LN1 = nn.LayerNorm(self.hidden_dim)
        self.LN2 = nn.LayerNorm(self.hidden_dim)
        self.activation = activation
        self.regularization = regularization
        self.r_se = r_se
        self.use_max_pooling = use_max_pooling
        self.block_index = 0          # set by MlpMixer; selects this block's dropout sites
        self.precision = None         # None: functional.get_precision(); "fp32" | "tf32" (not a reference argument)
        self._calls = 0

    def kernel_params(self):
        """Parameter tensors in the order of ``MmxMlpBlockParams`` (include/mmx.h)."""
        t, c = self.mlp_block_token_mixing, self.mlp_block_channel_mixing
        se = [self.se.excitation[0].weight, self.se.excitation[2].weight] if self.use_se else [None, None]
        return [self.LN1.weight, self.LN1.bias, t.fc1.weight, t.fc1.bias, t.fc2.weight, t.fc2.bias,
                self.LN2.weight, self.LN2.bias, c.fc1.weight, c.fc1.bias, c.fc2.weight, c.fc2.bias, *se]

    def bn_modules(self):
        """The four BatchNorm1d layers in execution order (regularization == -1)."""
        t, c = self.mlp_block_token_mixing, self.mlp_block_channel_mixing
        return [t.reg1, t.reg2, c.reg1, c.reg2]

    def meta(self, seed=0, step=0):
        p = self.regularization if self.regularization > 0.0 else 0.0
        return (self.tokens_mlp_dim, self.channels_mlp_dim, self.seq_len // self.r_se if self.use_se else 0,
                self.activation, self.use_se, self.use_max_pooling, self.training, self.block_index, p, seed, step,
                self.precision)

    def runners(self, B, device, need_backward, dropout=None):
        """This block's kernel runner: the stage-kernel chain with BatchNorm1d (regularization == -1, batch statistics), else
        the fused kernels.  ``dropout``: (seed, step, step_dev) of a static plan; None draws this call's own masks."""
        if self.regularization == -1.0:
            return [F_.MlpBnBlock(self, B, device, need_backward)]
        return [F_.FusedMixerBlock(self, B, device, need_backward, dropout or F_.dropout_source(self))]

    def forward(self, x):
        return F_.forward_layers(self, x)


class MlpMixer(nn.Module):
    """MotionMixer (mlp_mixer.py:239-337): embed -> num_blocks x MixerBlock -> LN -> conv_out -> fc_out."""

    def __init__(self, num_classes, num_blocks, hidden_dim, tokens_mlp_dim,
                 channels_mlp_dim, seq_len, pred_len, activation='gelu',
                 mlp_block_type='normal', regularization=0, input_size=51,
                 initialization='none', r_se=4, use_max_pooling=False,
                 use_se=False):
        super().__init__()
        self.num_classes = num_classes
        self.num_blocks = num_blocks
        self.hidden_dim = hidden_dim
        self.seq_len = seq_len
        self.tokens_mlp_dim = tokens_mlp_dim
        self.channels_mlp_dim = channels_mlp_dim
        self.input_size = input_size
        self.conv = nn.Conv2d(1, self.hidden_dim, (1, self.input_size), stride=1)
        self.activation = activation
        self.channel_only = False
        self.token_only = False
        self.Mixer_Block = nn.ModuleList(
            MixerBlock(self.tokens_mlp_dim, self.channels_mlp_dim, self.seq_len, self.hidden_dim,
                       activation=self.activation, regularization=regularization, initialization=initialization,
                       r_se=r_se, use_max_pooling=use_max_pooling, use_se=use_se)
            for _ in range(num_blocks))
        for i, mb in enumerate(self.Mixer_Block):
            mb.block_index = i
        self.LN = nn.LayerNorm(self.hidden_dim)
        self.fc_out = nn.Linear(self.hidden_dim, self.num_classes)
        self.pred_len = pred_len
        self.conv_out = nn.Conv1d(self.seq_len, self.pred_len, 1, stride=1)
        self.precision = None         # None: functional.get_precision(); set through set_precision()

    def set_precision(self, precision):
        """"fp32" (1e-5 parity, default) | "tf32" (tensor-core contractions inside the MixerBlocks, 2e-3 parity) | None
        (follow ``functional.set_precision``).  Not a reference argument: the constructor signature stays the reference's."""
        if precision is not None and precision not in F_.L.MMX_PREC:
            raise ValueError("unknown precision %r" % (precision,))
        self.precision = precision
        for mb in self.Mixer_Block:
            mb.precision = precision
        return self

    def runners(self, B, device, need_backward, dropout=None):
        """The kernel runners of one forward pass in order: embedding, blocks, head (see ``MixerBlock.runners``).  Yielded one
        at a time, so that ``model(x)`` builds each layer's runner just before the layer runs."""
        yield F_.LinearEmbed(self, B, device, need_backward)
        for mb in self.Mixer_Block:
            yield from mb.runners(B, device, need_backward, dropout)
        yield F_.MlpHead(self, B, device, need_backward)

    def forward(self, x):
        """x: [B, seq_len, input_size] -> [B, pred_len, num_classes]  (mlp_mixer.py:306-337)."""
        if x.dim() != 3 or x.shape[1] != self.seq_len or x.shape[2] != self.input_size:
            raise RuntimeError("MlpMixer.forward: expected [B, %d, %d], got %s" % (self.seq_len, self.input_size, tuple(x.shape)))
        return F_.forward_layers(self, x)
