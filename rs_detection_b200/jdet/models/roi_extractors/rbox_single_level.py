"""jdet.models.roi_extractors.rbox_single_level -- python/jdet/models/roi_extractors/rbox_single_level.py.

RboxSingleRoIExtractor: the v0 `ROIAlignRotated` layer (no -0.5 shift, counter-clockwise), levels mapped on the
RoI as given (`w_enlarge` / `h_enlarge` are stored and, like in the reference's execute (:80-104), never
applied).  Same fused launch as OrientedSingleRoIExtractor with `version = 0` and no extension.
"""
import torch
from torch import nn

from .... import core
from ...ops import roi_align_rotated
from .oriented_single_level import _FusedExtractFn


class RboxSingleRoIExtractor(nn.Module):
    def __init__(self, roi_layer, out_channels, featmap_strides, finest_scale=56, w_enlarge=1.2, h_enlarge=1.4):
        super(RboxSingleRoIExtractor, self).__init__()
        self.roi_layers = self.build_roi_layers(roi_layer, featmap_strides)
        self.out_channels = out_channels
        self.featmap_strides = featmap_strides
        self.finest_scale = finest_scale
        self.w_enlarge = w_enlarge
        self.h_enlarge = h_enlarge

    @property
    def num_inputs(self):
        return len(self.featmap_strides)

    def init_weights(self):
        pass

    def build_roi_layers(self, layer_cfg, featmap_strides):
        cfg = layer_cfg.copy()
        layer_type = cfg.pop('type')
        assert hasattr(roi_align_rotated, layer_type)  # :46-48: the layer is chosen BY NAME
        layer_cls = getattr(roi_align_rotated, layer_type)
        return nn.ModuleList([layer_cls(spatial_scale=1 / s, **cfg) for s in featmap_strides])

    def map_roi_levels(self, rois, num_levels):
        """(:53-71)"""
        scale = torch.sqrt(rois[:, 3] * rois[:, 4])
        target_lvls = torch.floor(torch.log2(scale / self.finest_scale + 1e-6))
        return target_lvls.clamp(min=0, max=num_levels - 1).long()

    def forward(self, feats, rois):
        if len(feats) == 1:
            return self.roi_layers[0](feats[0], rois)
        layer = self.roi_layers[0]
        cfg = core.make_roi_cfg([tuple(f.shape) for f in feats], [l.spatial_scale for l in self.roi_layers[:len(feats)]],
                                layer.output_size, int(layer.sampling_ratio), version=0, extend=(1.0, 1.0),
                                finest_scale=float(self.finest_scale))
        return _FusedExtractFn.apply(rois, cfg, layer.memory_format, *feats)

    execute = forward
