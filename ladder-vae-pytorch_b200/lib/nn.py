"""Kernel-backed mirror of the reference's lib/nn.py (ResidualBlock, ResidualGatedBlock,
GateLayer2d) plus the leaf modules they are built from.

Same class names, constructor arguments, ``nn.Sequential`` child indices (hence ``state_dict``
keys) and error behaviour as the reference (lib/nn.py:5-126).  Every parameter holder is still a
real ``nn.Conv2d`` / ``nn.BatchNorm2d`` submodule so forward hooks (boilr data-dependent init)
keep working: when a hook is registered anywhere inside a block the block runs module by module,
otherwise it runs the fused kernel sequence (BN+act pass -> conv with Dropout2d folded into its
epilogue -> ... -> gate * sigmoid + residual).
"""
from __future__ import annotations

import torch
from torch import nn

from lvae_b200 import ops


# ----------------------------------------------------------------------------- leaf modules
class Conv2d(nn.Conv2d):
    """nn.Conv2d whose forward/backward run lvae_conv2d_gather / lvae_conv2d_wgrad."""

    def __init__(self, *args, **kwargs):
        super().__init__(*args, **kwargs)
        k, s, p = self.kernel_size, self.stride, self.padding
        if self.groups != 1 or self.dilation != (1, 1) or k[0] != k[1] or s[0] != s[1] or p[0] != p[1] \
                or self.padding_mode != "zeros":
            raise NotImplementedError("lvae_b200.Conv2d supports square, ungrouped, undilated, zero-padded convs")
        self.spec = ops.ConvSpec(self.out_channels, self.in_channels, k[0], s[0], p[0])

    def forward(self, x, x2=None, out_scale=None, res=None, stats_bn=None, x_lowp=None):
        ops.note_conv_call(bool(self._forward_hooks))
        return ops.conv2d(x, self.weight, self.bias, self.spec, x2=x2, out_scale=out_scale, res=res, stats_bn=stats_bn,
                          x_lowp=x_lowp)


class ConvTranspose2d(nn.ConvTranspose2d):
    def __init__(self, *args, **kwargs):
        super().__init__(*args, **kwargs)
        k, s, p, op = self.kernel_size, self.stride, self.padding, self.output_padding
        if self.groups != 1 or self.dilation != (1, 1) or k[0] != k[1] or s[0] != s[1] or p[0] != p[1] or op[0] != op[1]:
            raise NotImplementedError("lvae_b200.ConvTranspose2d supports square, ungrouped, undilated convs")
        self.spec = ops.ConvSpec(self.out_channels, self.in_channels, k[0], s[0], p[0], transposed=True,
                                 output_padding=op[0])

    def forward(self, x, out_scale=None, res=None):
        ops.note_conv_call(bool(self._forward_hooks))
        return ops.conv2d(x, self.weight, self.bias, self.spec, out_scale=out_scale, res=res)


class BatchNorm2d(nn.BatchNorm2d):
    """nn.BatchNorm2d on lvae_bn_* kernels (batch statistics in train(), running ones in eval())."""

    def stat_acc(self, device):
        acc = getattr(self, "_stat_acc", None)
        if acc is None or acc.device != device:
            acc = torch.zeros(ops.BN_STRIPES * 2 * self.num_features, dtype=torch.float64, device=device)
            self._stat_acc = acc
        return acc

    def forward(self, x):
        return ops.bn_act(x, self, 0)


class _Nonlin(nn.Module):
    act_id = 0

    def forward(self, x):
        return ops.bn_act(x, None, self.act_id)


class ReLU(_Nonlin):
    act_id = 1


class LeakyReLU(_Nonlin):
    act_id = 2


class ELU(_Nonlin):
    act_id = 3


class SELU(_Nonlin):
    act_id = 4


NONLIN = {"relu": ReLU, "leakyrelu": LeakyReLU, "elu": ELU, "selu": SELU}
_TORCH_NONLIN = {nn.ReLU: ReLU, nn.LeakyReLU: LeakyReLU, nn.ELU: ELU, nn.SELU: SELU}


def resolve_nonlin(nonlin):
    """Accept our classes, the torch classes the reference passes around, or a name."""
    if isinstance(nonlin, str):
        return NONLIN[nonlin]
    return _TORCH_NONLIN.get(nonlin, nonlin)


class Dropout2d(nn.Module):
    """Channel dropout.  Inside a fused block the mask is folded into the preceding conv's
    epilogue; standalone (hooked / non-default block orders) it multiplies directly."""

    def __init__(self, p=0.5):
        super().__init__()
        if p is None or p < 0 or p > 1:      # nn.Dropout2d(None) raises too (lib/nn.py:89)
            raise TypeError("dropout probability has to be between 0 and 1, but got {}".format(p))
        self.p = float(p)

    def mask(self, x):
        if not self.training or self.p == 0.0:
            return None
        return ops.next_mask(x.shape[0], x.shape[1], self.p, x.device)

    def forward(self, x):
        m = self.mask(x)
        return x if m is None else x * m.view(x.shape[0], x.shape[1], 1, 1).to(x.dtype)

    def extra_repr(self):
        return "p={}".format(self.p)


class Interpolate(nn.Module):
    """boilr.nn.Interpolate(scale=2): bilinear, align_corners=False (models/lvae.py:144)."""

    def __init__(self, size=None, scale=None, mode="bilinear", align_corners=False):
        super().__init__()
        if scale != 2 or size is not None or mode != "bilinear" or align_corners:
            raise NotImplementedError("lvae_b200.Interpolate implements bilinear x2, align_corners=False")
        self.scale = scale

    def forward(self, x):
        return ops.upsample2x(x)


def _hooked(module: nn.Module) -> bool:
    for m in module.modules():
        if m._forward_hooks or m._forward_pre_hooks or m._backward_hooks:
            return True
    return False


# ----------------------------------------------------------------------------- reference classes
class GateLayer2d(nn.Module):
    """1x1 conv C -> 2C, then nonlin(first half) * sigmoid(second half)  (lib/nn.py:108-126)."""

    def __init__(self, channels, kernel_size, nonlin=LeakyReLU):
        super().__init__()
        assert kernel_size % 2 == 1
        self.conv = Conv2d(channels, 2 * channels, kernel_size, padding=kernel_size // 2)
        self.nonlin = resolve_nonlin(nonlin)()

    def forward(self, x, res=None):
        return ops.gate(self.conv(x), res, getattr(self.nonlin, "act_id", 0))


class ResidualBlock(nn.Module):
    """out = gate(f(x)) + x with f laid out by ``block_type`` (lib/nn.py:5-99):
    a = activation, b = batch norm, c = conv, d = dropout."""

    default_kernel_size = (3, 3)

    def __init__(self, channels, nonlin, kernel=None, groups=1, batchnorm=True, block_type=None, dropout=None,
                 gated=None):
        super().__init__()
        if kernel is None:
            kernel = self.default_kernel_size
        elif isinstance(kernel, int):
            kernel = (kernel, kernel)
        elif len(kernel) != 2:
            raise ValueError("kernel has to be None, int, or an iterable of length 2")
        assert all(k % 2 == 1 for k in kernel), "kernel sizes have to be odd"
        nonlin = resolve_nonlin(nonlin)
        self.gated = gated
        layers = []
        conv = lambda i: Conv2d(channels, channels, kernel[i], padding=kernel[i] // 2, groups=groups)
        if block_type == "cabdcabd":
            for i in (0, 1):
                layers += [conv(i), nonlin()]
                if batchnorm:
                    layers.append(BatchNorm2d(channels))
                if dropout is not None:
                    layers.append(Dropout2d(dropout))
        elif block_type == "bacdbac":
            for i in (0, 1):
                if batchnorm:
                    layers.append(BatchNorm2d(channels))
                layers += [nonlin(), conv(i)]
                if dropout is not None and i == 0:
                    layers.append(Dropout2d(dropout))
        elif block_type == "bacdbacd":
            for i in (0, 1):
                if batchnorm:
                    layers.append(BatchNorm2d(channels))
                layers += [nonlin(), conv(i), Dropout2d(dropout)]
        else:
            raise ValueError("unrecognized block type '{}'".format(block_type))
        if gated:
            layers.append(GateLayer2d(channels, 1, nonlin))
        self.block = nn.Sequential(*layers)
        self._plan = self._make_plan(list(self.block))
        self._whole_block = self.takes_block_node(self._plan)

    @staticmethod
    def takes_block_node(plan) -> bool:
        """(BN, act, conv, [dropout]) x 2 [+ gate] -- 'bacdbacd' and 'bacdbac', gated or not, with a Dropout2d behind either
        conv, both or neither, and the same activation in both BatchNorm + activation steps -- runs as ONE autograd node
        with a hand-made backward (ops.residual_block).  'cabdcabd' and batchnorm=False run step by step."""
        kinds = [k for k, _, _ in plan]
        return (kinds in (["bnact", "conv", "bnact", "conv"], ["bnact", "conv", "bnact", "conv", "gate"])
                and plan[0][1] is not None and plan[2][1] is not None and plan[0][2] == plan[2][2])

    @staticmethod
    def _make_plan(mods):
        """Greedy fusion of the Sequential into kernel steps."""
        plan, i = [], 0
        while i < len(mods):
            m = mods[i]
            nxt = mods[i + 1] if i + 1 < len(mods) else None
            if isinstance(m, BatchNorm2d):
                if isinstance(nxt, _Nonlin):
                    plan.append(("bnact", m, nxt.act_id))
                    i += 2
                else:
                    plan.append(("bnact", m, 0))
                    i += 1
            elif isinstance(m, _Nonlin):
                plan.append(("bnact", None, m.act_id))
                i += 1
            elif isinstance(m, Conv2d):
                if isinstance(nxt, Dropout2d):
                    plan.append(("conv", m, nxt))
                    i += 2
                else:
                    plan.append(("conv", m, None))
                    i += 1
            elif isinstance(m, Dropout2d):
                plan.append(("drop", m, None))
                i += 1
            elif isinstance(m, GateLayer2d):
                plan.append(("gate", m, None))
                i += 1
            else:
                raise TypeError("unexpected module in residual block: %r" % (m,))
        return plan

    def forward(self, x):
        if _hooked(self):
            return self.block(x) + x
        if self._whole_block and ops.whole_block_enabled():
            p = self._plan
            return ops.residual_block(x, p[0][1], p[1][1], p[1][2], p[2][1], p[3][1], p[3][2], p[4][1] if len(p) == 5 else None,
                                      p[0][2])
        h, last = x, len(self._plan) - 1
        for idx, (kind, m, aux) in enumerate(self._plan):
            if kind == "bnact":
                h = ops.bn_act(h, m, aux)
            elif kind == "conv":
                mask = aux.mask(h) if aux is not None else None
                h = m(h, out_scale=mask, res=x if idx == last else None)
            elif kind == "drop":
                h = m(h)
            else:  # gate: always the last step
                h = m(h, res=x)
        if self._plan[last][0] not in ("conv", "gate"):
            h = h + x
        return h


class ResidualGatedBlock(ResidualBlock):

    def __init__(self, *args, **kwargs):
        super().__init__(*args, **kwargs, gated=True)
