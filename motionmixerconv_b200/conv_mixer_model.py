"""Drop-in replacement for the reference ``h36m/conv_mixer_model.py`` (``ConvMixer``) and
``conv_mixer/encoding/positional_encoder.py`` (``PoseEncoder``).

Same constructor arguments (conv_mixer_model.py:357-379), same ``forward(x)`` signature, same
``state_dict`` keys / shapes / registration order (including the aliased ``se2.*`` keys and the
``encoder.frequencies`` buffer), same default initialisation from the same ``torch.manual_seed`` (the
sub-modules are created in the reference's construction order so the RNG draws line up).  The
sub-modules are *parameter holders*: all arithmetic of ``forward`` runs in the fused sm_100a kernels
behind ``motionmixerconv_b200.functional`` — encoder, one kernel per ConvMixerBlock half, head.
"""
from __future__ import annotations

from typing import Tuple, Union

import os

import torch
import torch.nn as nn

from . import functional as F_


class PoseEncoder(nn.Module):
    """Parameter holder for positional_encoder.py:5-97 (harmonic embedding -> embed_mlp -> channelUpscaling)."""

    def __init__(self, dimPosIn, in_nTP, dimPosEmb, conv_nChan, n_harmonic_functions, omega0):
        super().__init__()
        self.n_harmonic_functions = n_harmonic_functions
        self.conv_nChan = conv_nChan
        if n_harmonic_functions <= 0:
            dimHarmonic = dimPosIn
        else:
            self.register_buffer('frequencies', omega0 * (2.0 ** torch.arange(n_harmonic_functions)))
            dimHarmonic = n_harmonic_functions * dimPosIn * 2
        self.embed_mlp = nn.Linear(dimHarmonic, dimPosEmb)
        self.channelUpscaling = nn.Linear(1, conv_nChan)

    def forward(self, x):
        """x: [bs, in_nTP, dimPosIn] -> [bs, conv_nChan, in_nTP, dimPosEmb]"""
        hn = max(int(self.n_harmonic_functions), 0)
        return F_.pose_encoder(x, hn, self.conv_nChan, self.frequencies if hn > 0 else None, self.embed_mlp.weight,
                               self.embed_mlp.bias, self.channelUpscaling.weight, self.channelUpscaling.bias)


class MultiChanSELayer(nn.Module):
    """Parameter holder for the squeeze-excitation over frames (conv_mixer_model.py:11-70)."""

    def __init__(self, in_nTP: int, r: int = 4, use_max_pooling: bool = False):
        super().__init__()
        self.squeezeBlock = nn.AdaptiveAvgPool2d((1, 1)) if not use_max_pooling else nn.AdaptiveMaxPool2d((1, 1))
        self.excitationBlock = nn.Sequential(
            nn.Linear(in_nTP, in_nTP // r, bias=False),
            nn.ReLU(inplace=True),
            nn.Linear(in_nTP // r, in_nTP, bias=False),
            nn.Sigmoid()
        )

    def forward(self, x):
        raise NotImplementedError("MultiChanSELayer is fused into ConvMixerBlock.forward (no standalone kernel)")


def _same_pad(k):
    return (k - 1) // 2        # PyTorch padding='same': the surplus of an even kernel goes to the bottom / right


class ConvBlock(nn.Module):
    """Parameter holder for conv -> act -> reg (conv_mixer_model.py:73-142)."""

    def __init__(self, batchnorm_dim: int, conv_in_chan: int = 1, conv_out_chan: int = 1,
                 conv_kernel_shape: Tuple[int, int] = (1, 3), conv_stride: Tuple[int, int] = (1, 1),
                 conv_padding: Union[Tuple[int, int], str] = "same", activation: str = 'gelu', regularization: float = 0.0):
        super().__init__()
        self.bn_dim = batchnorm_dim
        self.conv = nn.Conv2d(conv_in_chan, conv_out_chan, conv_kernel_shape, stride=conv_stride, padding=conv_padding)
        if regularization > 0.0:
            self.reg = nn.Dropout(regularization)
        elif regularization == -1.0:
            self.reg = nn.BatchNorm2d(self.bn_dim)
        else:
            self.reg = nn.Identity()
        if activation == 'gelu':
            self.act = nn.GELU()
        elif activation == 'mish':
            self.act = nn.Mish()
        else:
            raise ValueError('Unknown activation function type: %s' % activation)
        self.activation = activation
        self.regularization = regularization
        kt, kp = self.conv.kernel_size
        if tuple(self.conv.stride) != (1, 1):
            raise NotImplementedError("ConvBlock: only stride (1,1) is built (the residual add of ConvMixerBlock needs it)")
        if isinstance(conv_padding, str):
            if conv_padding != "same":
                raise NotImplementedError("ConvBlock: padding must be 'same' or a tuple keeping the [T,E] shape")
            self.pad = (_same_pad(kt), _same_pad(kp))
        else:
            pt, pp = conv_padding
            # a padding that changes the [in_nTP, dimPosEmb] shape constructs fine in the reference and fails in
            # forward at the residual add (conv_mixer_model.py:284); same here
            self.pad = (pt, pp) if (2 * pt == kt - 1 and 2 * pp == kp - 1) else None
        self.kernel = (kt, kp)

    def forward(self, x):
        raise NotImplementedError("ConvBlock is fused into ConvMixerBlock.forward (no standalone kernel)")


class ConvMixerBlock(nn.Module):
    """conv_mixer_model.py:145-292: one fused kernel per half (LN -> conv -> act -> reg -> SE -> +res)."""

    def __init__(self, dimPosEmb: int, in_nTP: int, conv_nChan: int, conv1_kernel_shape: Tuple[int, int] = (1, 3),
                 conv1_stride=None, conv1_padding=None, mode_conv: str = "twice", conv2_kernel_shape=None,
                 conv2_stride=None, conv2_padding=None, activation: str = 'gelu', regularization: float = 0,
                 use_se: bool = True, r_se: int = 4, use_max_pooling: bool = False):
        super().__init__()
        self.conv_nChan = conv_nChan
        self.in_nTP = in_nTP
        self.dimPosEmb = dimPosEmb
        self.mode_conv = mode_conv
        if conv1_padding is None:
            conv1_padding = "same"
        if conv1_stride is None:
            conv1_stride = (1, 1)
        self.conv1 = ConvBlock(batchnorm_dim=self.conv_nChan, conv_in_chan=self.conv_nChan, conv_out_chan=self.conv_nChan,
                               conv_kernel_shape=conv1_kernel_shape, conv_stride=conv1_stride, conv_padding=conv1_padding,
                               activation=activation, regularization=regularization)
        if use_se:
            self.se = MultiChanSELayer(self.in_nTP, r=r_se, use_max_pooling=use_max_pooling)
        else:
            self.se = nn.Identity()
        self.LN1 = nn.LayerNorm(self.dimPosEmb)
        if mode_conv == "twice":
            if conv2_kernel_shape is None:
                conv2_kernel_shape = (min(conv1_kernel_shape[1], in_nTP), min(conv1_kernel_shape[0], dimPosEmb))
            if conv2_stride is None:
                conv2_stride = (1, 1)
            if conv2_padding is None:
                conv2_padding = "same"
            self.conv2 = ConvBlock(batchnorm_dim=self.conv_nChan, conv_in_chan=self.conv_nChan, conv_out_chan=self.conv_nChan,
                                   conv_kernel_shape=conv2_kernel_shape, conv_stride=conv2_stride, conv_padding=conv2_padding,
                                   activation=activation, regularization=regularization)
            self.se2 = self.se
            self.LN2 = nn.LayerNorm(self.dimPosEmb)
        elif mode_conv == "once":
            self.conv2 = nn.Identity()
            self.se2 = nn.Identity()
            self.LN2 = nn.Identity()
        else:
            raise ValueError("mode_conv %s" % mode_conv + " must be one of 'once' or 'twice'")
        self.use_se = use_se
        self.r_se = r_se
        self.use_max_pooling = use_max_pooling
        self.activation = activation
        self.regularization = regularization
        self.block_index = 0      # set by ConvMixer; selects this block's dropout sites
        self.precision = None     # None / "fp32" | "tf32"; set through ConvMixer.set_precision (not a reference argument)
        self._calls = 0

    # ---- kernel plumbing -----------------------------------------------------------------------
    def se_weights(self):
        if not self.use_se:
            return [None, None]
        return [self.se.excitationBlock[0].weight, self.se.excitationBlock[2].weight]

    def half_params(self, half):
        """Parameter tensors in the order of ``MmxConvHalfParams`` (include/mmx.h)."""
        ln, cb = (self.LN1, self.conv1) if half == 0 else (self.LN2, self.conv2)
        return [ln.weight, ln.bias, cb.conv.weight, cb.conv.bias, *self.se_weights()]

    def half_meta(self, half, seed=0, step=0):
        cb = self.conv1 if half == 0 else self.conv2
        if cb.pad is None:
            raise RuntimeError("The size of tensor a must match the size of tensor b: conv padding %s with kernel %s does "
                               "not keep the [in_nTP, dimPosEmb] shape needed by the residual add" % (cb.conv.padding, cb.kernel))
        p = self.regularization if self.regularization > 0.0 else 0.0
        return (cb.kernel, cb.pad, self.in_nTP // self.r_se if self.use_se else 0, self.activation, self.use_se,
                self.use_max_pooling, self.training, 2 * self.block_index + half, p, seed, step)

    def uses_large_path(self, half, B):
        """True when this half runs as the stage-kernel chain instead of one fused kernel per direction."""
        if self.regularization == -1.0 and self.use_se and self.use_max_pooling:
            return True
        if os.environ.get("MMX_CONV_FORCE_LARGE", "0") == "1":     # tests: run any shape through the stage-kernel chain
            return True
        key = (half, B > 0)
        cache = self.__dict__.setdefault("_fits", {})
        if key not in cache:
            cache[key] = F_.conv_half_fits(max(B, 1), self.conv_nChan, self.in_nTP, self.dimPosEmb, self.half_meta(half))
        # Precision "tf32" leaves a half the fused fp32 kernels serve on them: chain + tcgen05 convolution measured slower at every
        # such cell (B200, 1000 W, B = 256 training steps, profiles/r2h_conv_tc5.jsonl): Optuna 5x5 at C = 8 (200 taps C*kt*kp)
        # 4.98 ms fused vs 5.10 ms chain (once), 8.10 vs 8.30 (twice); K3 (C = 4, 5x9 / 9x5, 180 taps) rollout training 22.8 vs
        # 31.5 ms.  The halves that already take the chain gain 1.6x (5x9) to 3.2x (9x29) from it.
        return not cache[key]

    def uses_tc5_conv(self, half, B):
        """True when, in precision "tf32", this half's convolutions run on tcgen05 once the half takes the stage-kernel chain."""
        key = (half, B > 0)
        cache = self.__dict__.setdefault("_tc5", {})
        if key not in cache:
            cache[key] = F_.conv_tc5_serves(max(B, 1), self.conv_nChan, self.in_nTP, self.dimPosEmb, self.half_meta(half))
        return self.precision == "tf32" and cache[key]

    def _half(self, x, half, seed, step):
        cb = self.conv1 if half == 0 else self.conv2
        meta, params = self.half_meta(half, seed, step), self.half_params(half)
        if self.uses_large_path(half, x.shape[0]):
            # shapes the fused kernels do not hold in shared memory (most of the Optuna grid at C = 8, E = 192) and BatchNorm
            # with the max squeeze: the same arithmetic as a chain of stage kernels (functional.ConvHalfLarge)
            return F_.conv_half_large(x, meta, params, cb.reg if self.regularization == -1.0 else None, self.precision)
        if self.regularization == -1.0:
            if self.training:
                return F_.conv_half_bn(x, meta, cb.reg, params)
            return F_.conv_half(x, meta, params, bn_aff=F_.bn_eval_affine(cb.reg))
        return F_.conv_half(x, meta, params)

    def forward(self, x: torch.Tensor):
        seed = step = 0
        if self.training and self.regularization > 0.0:
            seed = torch.initial_seed() & 0xFFFFFFFFFFFFFFFF
            step = self._calls
            self._calls = (self._calls + 1) & 0xFFFFFFFF
        x = self._half(x, 0, seed, step)
        if self.mode_conv == "twice":
            return self._half(x, 1, seed, step)
        # mode_conv="once": LN2 / conv2 are Identity but self.se is still applied (conv_mixer_model.py:287-292)
        s1, s2 = self.se_weights()
        return F_.se_tail(x, self.in_nTP // self.r_se if self.use_se else 0, self.use_se, self.use_max_pooling, s1, s2)


class ConvMixer(nn.Module):
    """conv_mixer_model.py:295-465: encoder -> num_blocks x ConvMixerBlock -> LN -> conv_out -> project_channels -> GELU -> fc_out."""

    def __init__(self, num_blocks: int, dimPosIn: int, dimPosEmb: int, dimPosOut: int, in_nTP: int, out_nTP: int,
                 conv_nChan: int = 1, conv1_kernel_shape: Tuple[int, int] = (1, 3), conv1_stride: Tuple[int, int] = (1, 1),
                 conv1_padding: Union[Tuple[int, int], None] = None, mode_conv: str = "twice",
                 conv2_kernel_shape: Union[Tuple[int, int], None] = None, conv2_stride: Union[Tuple[int, int], None] = None,
                 conv2_padding: Union[Tuple[int, int], None] = None, activation: str = 'gelu', regularization: float = 0,
                 use_se: bool = False, r_se: int = 4, use_max_pooling: bool = False,
                 encoder_n_harmonic_functions: int = 64, encoder_omega0: float = 0.1):
        super().__init__()
        self.dimPosIn = dimPosIn
        self.dimPosOut = dimPosOut
        self.dimPosEmb = dimPosEmb
        self.num_blocks = num_blocks
        self.in_nTP = in_nTP
        self.conv_nChan = conv_nChan
        self.activation = activation
        self.encoder = PoseEncoder(dimPosIn=self.dimPosIn, in_nTP=self.in_nTP, dimPosEmb=self.dimPosEmb,
                                   conv_nChan=self.conv_nChan, n_harmonic_functions=encoder_n_harmonic_functions,
                                   omega0=encoder_omega0)
        self.Mixer_Block = nn.ModuleList(
            ConvMixerBlock(dimPosEmb=self.dimPosEmb, in_nTP=self.in_nTP, conv_nChan=self.conv_nChan,
                           conv1_kernel_shape=conv1_kernel_shape, conv1_stride=conv1_stride, conv1_padding=conv1_padding,
                           mode_conv=mode_conv, conv2_kernel_shape=conv2_kernel_shape, conv2_stride=conv2_stride,
                           conv2_padding=conv2_padding, activation=activation, regularization=regularization,
                           use_se=use_se, r_se=r_se, use_max_pooling=use_max_pooling)
            for _ in range(num_blocks))
        for i, mb in enumerate(self.Mixer_Block):
            mb.block_index = i
        self.LN = nn.LayerNorm(self.dimPosEmb)
        self.out_nTP = out_nTP
        self.project_channels = nn.Conv2d(self.conv_nChan, 1, kernel_size=(1, 1), stride=1)
        self.conv_out = nn.Conv2d(in_channels=self.in_nTP, out_channels=self.out_nTP, kernel_size=1, stride=1)
        self.fc_out = nn.Linear(self.dimPosEmb, self.dimPosOut)
        self.precision = None         # fp32; set through set_precision()

    def set_precision(self, precision):
        """"fp32" / None (1e-5 parity, the default) | "tf32": the ConvBlock convolutions of the halves that run as the stage-kernel
        chain use the tensor cores (tcgen05, bf16x3; 2e-3 parity) where mmx_conv2d_tc5_serves.  Halves the fused fp32 kernels
        serve stay on them (faster, see ``ConvMixerBlock.uses_large_path``); the encoder and head stay fp32.  None does NOT follow
        ``functional.set_precision`` / MMX_PRECISION: the ConvMixer opts in here only.  Not a reference argument and not part of
        the state_dict.  Returns self."""
        if precision is not None and precision not in F_.L.MMX_PREC:
            raise ValueError("unknown precision %r" % (precision,))
        self.precision = precision
        for mb in self.Mixer_Block:
            mb.precision = precision
        return self

    def head_params(self):
        """Parameter tensors in the order of ``MmxConvHeadParams`` (include/mmx.h)."""
        return [self.LN.weight, self.LN.bias, self.conv_out.weight, self.conv_out.bias, self.project_channels.weight,
                self.project_channels.bias, self.fc_out.weight, self.fc_out.bias]

    def forward(self, x: torch.Tensor):
        """x: [batch_size, in_nTP, dimPosIn] -> [batch_size, out_nTP, dimPosOut]  (conv_mixer_model.py:428-465)."""
        if x.dim() != 3 or x.shape[1] != self.in_nTP or x.shape[2] != self.dimPosIn:
            raise RuntimeError("ConvMixer.forward: expected [B, %d, %d], got %s" % (self.in_nTP, self.dimPosIn, tuple(x.shape)))
        y = self.encoder(x)
        for mb in self.Mixer_Block:
            y = mb(y)
        return F_.conv_head(y, *self.head_params())
