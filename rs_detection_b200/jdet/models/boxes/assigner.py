"""jdet.models.boxes.assigner -- python/jdet/models/boxes/assigner.py:7-170 (MaxIoUAssigner).

`assign_wrt_overlaps` is one kernel (column max/argmax + thresholds + optional low-quality matching)
instead of ~10 small Jittor ops and a Python loop over GTs with `jt.sync_all()` every 100 (:152-160).
With the horizontal calculator `BboxOverlaps2D` (the oriented RPN's), `assign` takes `core.assign_hbb`, which gives
the same bits without storing the (num_gts, n) overlaps matrix, at every number of GTs.
"""
import torch

from .... import core
from ...ops._io import back, dev
from .iou_calculator import BboxOverlaps2D, BboxOverlaps2D_rotated, BboxOverlaps2D_rotated_v1

_CALCULATORS = {'BboxOverlaps2D_rotated': BboxOverlaps2D_rotated, 'BboxOverlaps2D_rotated_v1': BboxOverlaps2D_rotated_v1,
                'BboxOverlaps2D': BboxOverlaps2D}


class AssignResult:
    """assigner.py:7-22"""

    def __init__(self, num_gts, gt_inds, max_overlaps, labels=None):
        self.num_gts = num_gts
        self.gt_inds = gt_inds
        self.max_overlaps = max_overlaps
        self.labels = labels

    def add_gt_(self, gt_labels):
        self_inds = torch.arange(1, len(gt_labels) + 1, dtype=self.gt_inds.dtype, device=self.gt_inds.device)
        self.gt_inds = torch.cat([self_inds, self.gt_inds])
        self.max_overlaps = torch.cat([torch.ones((self.num_gts,), device=self.max_overlaps.device), self.max_overlaps])
        if self.labels is not None:
            self.labels = torch.cat([gt_labels.to(self.labels.dtype), self.labels])


class MaxIoUAssigner:
    def __init__(self, pos_iou_thr, neg_iou_thr, min_pos_iou=.0, gt_max_assign_all=True, ignore_iof_thr=-1,
                 ignore_wrt_candidates=True, match_low_quality=True, assigned_labels_filled=0,
                 iou_calculator=dict(type='BboxOverlaps2D_rotated_v1')):
        self.pos_iou_thr = pos_iou_thr
        self.neg_iou_thr = neg_iou_thr
        self.min_pos_iou = min_pos_iou
        self.gt_max_assign_all = gt_max_assign_all
        self.ignore_iof_thr = ignore_iof_thr
        self.ignore_wrt_candidates = ignore_wrt_candidates
        self.match_low_quality = match_low_quality
        self.assigned_labels_filled = assigned_labels_filled
        self.iou_calculator = _CALCULATORS[iou_calculator['type']]() if isinstance(iou_calculator, dict) else iou_calculator

    def assign(self, bboxes, gt_bboxes, gt_bboxes_ignore=None, gt_labels=None):
        if bboxes.shape[0] == 0 or gt_bboxes.shape[0] == 0:
            raise ValueError('No gt or bboxes')
        if isinstance(self.iou_calculator, BboxOverlaps2D):
            return self._assign_hbb(bboxes, gt_bboxes, gt_bboxes_ignore, gt_labels)
        overlaps = self.iou_calculator(gt_bboxes, bboxes)
        if (self.ignore_iof_thr > 0) and (gt_bboxes_ignore is not None) and (gt_bboxes_ignore.numel() > 0):
            raise NotImplementedError("'iof' ignore regions are not on the rotated hot path (the rotated "
                                      "calculators assert mode == 'iou', iou_calculator.py:108,148)")
        return self.assign_wrt_overlaps(overlaps, gt_labels)

    def _assign_hbb(self, bboxes, gt_bboxes, gt_bboxes_ignore, gt_labels):
        """assign_wrt_overlaps(BboxOverlaps2D()(gt_bboxes, bboxes)) in one fused call (rsdet_assign_hbb)."""
        if (self.ignore_iof_thr > 0) and (gt_bboxes_ignore is not None) and (gt_bboxes_ignore.numel() > 0):
            raise NotImplementedError("'iof' ignore regions are not supported by the fused horizontal assignment")
        assert gt_bboxes.size(-1) in [4, 5] and bboxes.size(-1) in [4, 5]
        anchors, fl = dev(bboxes[..., :4])
        gts, _ = dev(gt_bboxes[..., :4])
        gl = None if gt_labels is None else dev(gt_labels, torch.int32)[0]
        gt_inds, max_overlaps, labels = core.assign_hbb(
            gts.reshape(-1, 4), anchors.reshape(-1, 4), float(self.pos_iou_thr), self.neg_iou_thr, float(self.min_pos_iou),
            bool(self.match_low_quality), bool(self.gt_max_assign_all), gl, int(self.assigned_labels_filled))
        return AssignResult(gts.shape[0], back(gt_inds, fl), back(max_overlaps, fl), labels=back(labels, fl))

    def assign_wrt_overlaps(self, overlaps, gt_labels=None):
        if overlaps.numel() == 0:
            raise ValueError('No gt or proposals')
        num_gts = overlaps.size(0)
        ov = overlaps if overlaps.is_cuda else overlaps.cuda()
        gl = None if gt_labels is None else (gt_labels if gt_labels.is_cuda else gt_labels.cuda())
        gt_inds, max_overlaps, labels = core.assign_wrt_overlaps(
            ov, float(self.pos_iou_thr), self.neg_iou_thr, float(self.min_pos_iou), bool(self.match_low_quality),
            bool(self.gt_max_assign_all), gl, int(self.assigned_labels_filled))
        if not overlaps.is_cuda:
            gt_inds, max_overlaps = gt_inds.cpu(), max_overlaps.cpu()
            labels = None if labels is None else labels.cpu()
        return AssignResult(num_gts, gt_inds, max_overlaps, labels=labels)
