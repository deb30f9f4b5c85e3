"""jdet.ops.roi_align_rotated_v1 -- python/jdet/ops/roi_align_rotated_v1.py:300-373.

`ROIAlignRotated_v1(output_size, spatial_scale, sampling_ratio=0)` is looked up BY NAME from the
configs (`getattr(roi_align_rotated_v1, layer_type)`, oriented_single_level.py:43-51), so class name,
constructor arguments, the `output_size` tuple attribute and `__repr__` are kept verbatim.

Layouts (no reference counterpart).  Channels_last inputs are read without a layout copy and get channels_last
gradients.  `memory_format=torch.channels_last` (keyword of `roi_align` and of the layer, and so of a `roi_layer`
config dict) makes the kernel write a channels_last (K, C, ph, pw) output: a head that flattens it with `.view(K, -1)`
needs the default.  The values never depend on a layout.
"""
import warnings

import torch
from torch import nn

from ... import core

__all__ = ["ROIAlign"]  # sic, roi_align_rotated_v1.py:5


def _pair(x):
    return tuple(x) if isinstance(x, (tuple, list)) else (x, x)


def _grad_dtype(dtype):
    """fp16 / bf16 inputs are read natively and get their gradient in their own dtype; the rest is handled in fp32."""
    return dtype if dtype in (torch.float16, torch.bfloat16) else torch.float32


def _out_channels_last(memory_format):
    """Whether a `memory_format` argument asks for a channels_last RoI output; ValueError for anything but
    torch.contiguous_format and torch.channels_last."""
    if memory_format is torch.channels_last:
        return True
    if memory_format is torch.contiguous_format:
        return False
    raise ValueError(f"RoIAlignRotated: memory_format must be torch.contiguous_format or torch.channels_last, got {memory_format!r}")


def _maps_format(feats):
    """The layout of the gradient maps: the inputs' own when every level is channels_last."""
    return torch.channels_last if core.roi_maps_channels_last(feats) else torch.contiguous_format


def _deterministic_backward(cfg, op):
    """Whether the backward of `op` runs the ordered (bitwise reproducible) kernel: under
    `torch.use_deterministic_algorithms(True)`.  The adaptive sampling grid (sampling_ratio <= 0) has no deterministic
    kernel; like torch's own ops it then raises RuntimeError, or with `warn_only=True` warns and runs the atomic one."""
    if not torch.are_deterministic_algorithms_enabled():
        return False
    if cfg.sampling_ratio > 0:
        return True
    msg = (f"{op} backward with sampling_ratio <= 0 (adaptive sampling grid) does not have a deterministic implementation, "
           "but you set 'torch.use_deterministic_algorithms(True)'. You can turn off determinism just for this operation, "
           "or you can use the 'warn_only=True' option, if that's acceptable for your application. You can also use a "
           "fixed sampling_ratio > 0, whose backward is deterministic.")
    if torch.is_deterministic_algorithms_warn_only_enabled():
        warnings.warn(msg, UserWarning)
        return False
    raise RuntimeError(msg)


class _RotatedROIAlignFn(torch.autograd.Function):
    """Forward + backward of one feature map (the reference's jt.Function, :300-351); rois get no grad.  The output is
    fp32 whatever the input's dtype, like the reference's float kernels."""

    @staticmethod
    def forward(ctx, input, rois, output_size, spatial_scale, sampling_ratio, version, memory_format=torch.contiguous_format):
        assert rois.shape[1] == 6
        cfg = core.make_roi_cfg([tuple(input.shape)], [spatial_scale], output_size, int(sampling_ratio), version)
        ctx.cfg, ctx.shape, ctx.dtype = cfg, tuple(input.shape), _grad_dtype(input.dtype)
        ctx.maps_format = _maps_format([input])
        ctx.save_for_backward(rois)
        return core.roi_align_rotated_forward(cfg, [input], rois, memory_format=memory_format)

    @staticmethod
    def backward(ctx, grad_output):
        (rois,) = ctx.saved_tensors
        det = _deterministic_backward(ctx.cfg, "ROIAlignRotated_v1" if ctx.cfg.version == 1 else "ROIAlignRotated")
        grads = core.roi_align_rotated_backward(ctx.cfg, grad_output, rois, [ctx.shape], feat_dtype=ctx.dtype,
                                                deterministic=det, memory_format=ctx.maps_format)
        return grads[0], None, None, None, None, None, None


def roi_align(input, rois, output_size, spatial_scale, sampling_ratio, memory_format=torch.contiguous_format):
    _out_channels_last(memory_format)
    return _RotatedROIAlignFn.apply(input, rois, _pair(output_size), spatial_scale, sampling_ratio, 1, memory_format)


def _layer_repr(layer):
    tmpstr = layer.__class__.__name__ + "("
    tmpstr += "output_size=" + str(layer.output_size)
    tmpstr += ", spatial_scale=" + str(layer.spatial_scale)
    tmpstr += ", sampling_ratio=" + str(layer.sampling_ratio)
    if layer.memory_format is not torch.contiguous_format:
        tmpstr += ", memory_format=" + str(layer.memory_format)
    tmpstr += ")"
    return tmpstr


class ROIAlignRotated_v1(nn.Module):
    def __init__(self, output_size, spatial_scale, sampling_ratio=0, memory_format=torch.contiguous_format):
        super(ROIAlignRotated_v1, self).__init__()
        self.output_size = _pair(output_size)
        self.spatial_scale = spatial_scale
        self.sampling_ratio = sampling_ratio
        _out_channels_last(memory_format)
        self.memory_format = memory_format

    def forward(self, input, rois):
        return roi_align(input, rois, self.output_size, self.spatial_scale, self.sampling_ratio, self.memory_format)

    execute = forward  # Jittor spelling

    __repr__ = _layer_repr
