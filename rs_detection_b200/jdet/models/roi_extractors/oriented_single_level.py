"""jdet.models.roi_extractors.oriented_single_level -- python/jdet/models/roi_extractors/oriented_single_level.py.

Same class name, constructor arguments and `execute(feats, rois, roi_scale_factor=None)` contract as
the reference's OrientedSingleRoIExtractor, but the body is ONE fused launch (RoI extension, level
mapping, per-level RoIAlignRotated and the scatter back into RoI order) instead of the reference's
Python loop over levels with boolean gathers / masked scatter-adds (:105-112).
"""
import torch
from torch import nn

from .... import core
from ...ops import roi_align_rotated_v1
from ...ops.roi_align_rotated_v1 import _deterministic_backward, _grad_dtype, _maps_format


def _pair(x):
    return tuple(x) if isinstance(x, (tuple, list)) else (x, x)


class _FusedExtractFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, rois, cfg, memory_format, *feats):
        ctx.cfg = cfg
        ctx.shapes = [tuple(f.shape) for f in feats]
        ctx.dtype = _grad_dtype(feats[0].dtype)      # core rejects levels that mix fp16 / bf16 with another dtype
        ctx.maps_format = _maps_format(feats)
        ctx.save_for_backward(rois)
        return core.roi_align_rotated_forward(cfg, feats, rois, memory_format=memory_format)

    @staticmethod
    def backward(ctx, grad_output):
        (rois,) = ctx.saved_tensors
        det = _deterministic_backward(ctx.cfg, "RoI extractor (RoIAlignRotated)")
        grads = core.roi_align_rotated_backward(ctx.cfg, grad_output, rois, ctx.shapes, feat_dtype=ctx.dtype,
                                                deterministic=det, memory_format=ctx.maps_format)
        return (None, None, None, *grads)


class OrientedSingleRoIExtractor(nn.Module):
    """Extract RoI features from a single level feature map (each RoI is mapped to one FPN level by its
    extended scale).  Args as in the reference (:22-34).  The output layout is the roi layer's `memory_format`."""

    def __init__(self, roi_layer, out_channels, featmap_strides, extend_factor=(1., 1.), finest_scale=56):
        super(OrientedSingleRoIExtractor, self).__init__()
        self.roi_layers = self.build_roi_layers(roi_layer, featmap_strides)
        self.out_channels = out_channels
        self.featmap_strides = featmap_strides
        self.extend_factor = extend_factor
        self.finest_scale = finest_scale

    @property
    def num_inputs(self):
        return len(self.featmap_strides)

    def init_weights(self):
        pass

    def build_roi_layers(self, layer_cfg, featmap_strides):
        cfg = layer_cfg.copy()
        layer_type = cfg.pop('type')
        assert hasattr(roi_align_rotated_v1, layer_type)  # :46-48: the layer is chosen BY NAME
        layer_cls = getattr(roi_align_rotated_v1, layer_type)
        return nn.ModuleList([layer_cls(spatial_scale=1 / s, **cfg) for s in featmap_strides])

    def map_roi_levels(self, rois, num_levels):
        """(:53-71) level index of each RoI, computed by the same kernel that does the pooling."""
        scale = torch.sqrt(rois[:, 3] * rois[:, 4])
        target_lvls = torch.floor(torch.log2(scale / self.finest_scale + 1e-6))
        return target_lvls.clamp(min=0, max=num_levels - 1).long()

    def roi_rescale(self, rois, scale_factor):
        """(:73-89)"""
        if scale_factor is None:
            return rois
        h_scale_factor, w_scale_factor = _pair(scale_factor)
        new_rois = rois.clone()
        new_rois[:, 3] = w_scale_factor * new_rois[:, 3]
        new_rois[:, 4] = h_scale_factor * new_rois[:, 4]
        return new_rois

    def forward(self, feats, rois, roi_scale_factor=None):
        if len(feats) == 1:
            return self.roi_layers[0](feats[0], rois)  # :92-93 (no extension on this branch)
        layer = self.roi_layers[0]
        rois = self.roi_rescale(rois, roi_scale_factor) if roi_scale_factor is not None else rois
        # note: the reference rescales by extend_factor, maps levels on the extended box, THEN applies
        # roi_scale_factor (:100-103); roi_scale_factor is always None on the Oriented R-CNN path.  A
        # non-None value is folded in before the extension, which commutes for the RoI geometry but
        # would move the level boundaries -- rejected rather than silently different.
        if roi_scale_factor is not None:
            raise NotImplementedError("roi_scale_factor is unused on the Oriented R-CNN path")
        eh, ew = _pair(self.extend_factor)
        cfg = core.make_roi_cfg([tuple(f.shape) for f in feats], [l.spatial_scale for l in self.roi_layers[:len(feats)]],
                                layer.output_size, int(layer.sampling_ratio), version=1, extend=(eh, ew),
                                finest_scale=float(self.finest_scale))
        return _FusedExtractFn.apply(rois, cfg, layer.memory_format, *feats)

    execute = forward
