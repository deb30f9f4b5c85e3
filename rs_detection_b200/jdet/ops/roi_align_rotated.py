"""jdet.ops.roi_align_rotated -- python/jdet/ops/roi_align_rotated.py:256-329 (v0 convention: no -0.5
centre shift, counter-clockwise rotation; used by RboxSingleRoIExtractor)."""
import torch
from torch import nn

from .roi_align_rotated_v1 import _layer_repr, _out_channels_last, _pair, _RotatedROIAlignFn

__all__ = ["ROIAlign"]


def roi_align(input, rois, output_size, spatial_scale, sampling_ratio, memory_format=torch.contiguous_format):
    _out_channels_last(memory_format)
    return _RotatedROIAlignFn.apply(input, rois, _pair(output_size), spatial_scale, sampling_ratio, 0, memory_format)


class ROIAlignRotated(nn.Module):
    def __init__(self, output_size, spatial_scale, sampling_ratio=0, memory_format=torch.contiguous_format):
        super(ROIAlignRotated, self).__init__()
        self.output_size = _pair(output_size)
        self.spatial_scale = spatial_scale
        self.sampling_ratio = sampling_ratio
        _out_channels_last(memory_format)
        self.memory_format = memory_format

    def forward(self, input, rois):
        return roi_align(input, rois, self.output_size, self.spatial_scale, self.sampling_ratio, self.memory_format)

    execute = forward

    __repr__ = _layer_repr
