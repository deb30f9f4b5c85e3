"""Top-level `merge.py` of the reference: two-model FAIR1M CSV ensemble (merge.py:14-27, 54-156).

The horizontal NMS (`nms`, keeps `iou < thresh`) runs on the device: `merge_csv_with_class` /
`merge_csv_without_class` send EVERY (image, class) group of the ensemble through one launch of the
engine (`RSDET_NMS_HBB`, float64).  The ensemble converts its rows with `rsdet_poly2obb`, the device
restatement of the reference's `cv2.minAreaRect` + le90 step (merge.py:73-100), bit for bit; `obb2hbb`
stays numpy float64, whose `cos`/`sin` bits decide the NMS.  `poly2obb` below is the host OpenCV
function, kept as the reference for the device call.
"""
import numpy as np
import torch

from .. import core
from .._lib import NMS_HBB, require_cuda

FAIR1M_1_5_CLASSES = ['Airplane', 'Ship', 'Vehicle', 'Basketball_Court', 'Tennis_Court', 'Football_Field',
                      'Baseball_Field', 'Intersection', 'Roundabout', 'Bridge']


def nms(boxes, thresh):
    """boxes (n,5) float64 [x1,y1,x2,y2,score]; keeps `iou < thresh`; returns np.array of kept indices in
    descending-score order (merge.py:14-27)."""
    require_cuda()
    b = np.ascontiguousarray(boxes, dtype=np.float64).reshape(-1, 5)
    if b.shape[0] == 0:
        return np.array([], dtype=np.int64)
    t = torch.from_numpy(b).cuda()
    res = core.nms(NMS_HBB, t[:, :4], t[:, 4], float(thresh), want_mask=False, want_sorted=False, want_score=True,
                   ws_tag="merge")
    return res.score_idx.cpu().numpy()


def read_csv_to_numpy(submit_csvfile_path):
    """:54-70 -> (n,11) float64 [image id, 8 coords, score, class index (1-based)]"""
    rows = []
    with open(submit_csvfile_path, "r") as f:
        for line in f.readlines():
            sp = line.strip().split(",")
            assert len(sp) == 11, "csv file format error"
            assert sp[1] in FAIR1M_1_5_CLASSES, "laebl name not matched"
            rows.append([int(sp[0].split(".")[0]), *[float(x) for x in sp[2:-1]], float(sp[-1]),
                         FAIR1M_1_5_CLASSES.index(sp[1]) + 1])
    return np.array(rows)


def poly2obb(polys):
    """:73-100 (OpenCV minAreaRect, le90-style normalisation) -- the same code as jdet.ops.bbox_transforms.poly2obb."""
    from .ops.bbox_transforms import poly2obb as _p2o
    return _p2o(polys)


def obb2hbb(obboxes):
    """:103-112"""
    center, w, h, theta, _ = np.split(obboxes, [2, 3, 4, 5], axis=-1)
    Cos, Sin = np.cos(theta), np.sin(theta)
    bias = np.concatenate([np.abs(w / 2 * Cos) + np.abs(h / 2 * Sin), np.abs(w / 2 * Sin) + np.abs(h / 2 * Cos)], axis=-1)
    return np.concatenate([center - bias, center + bias], axis=-1)


def save_to_csv(data, output_path):
    """:114-124"""
    with open(output_path, "w") as f:
        for each in data:
            temp = [f"{int(each[0])}.tif", FAIR1M_1_5_CLASSES[int(each[10]) - 1]]
            temp += ["{:.4f}".format(i) for i in each[1:9]]
            temp.append("{:.4f}".format(each[9]))
            f.write(",".join(temp))
            f.write("\n")


def _grouped_nms(dets, group, thr_per_group):
    """dets (n,11), group (n,) int32 ascending-group output order; returns kept row indices ordered by
    (group asc, score desc)."""
    require_cuda()
    polys = torch.from_numpy(np.ascontiguousarray(dets[:, 1:9], dtype=np.float64)).cuda()
    hbb = obb2hbb(core.poly2obb(polys).cpu().numpy())
    b = torch.from_numpy(np.ascontiguousarray(hbb, dtype=np.float64)).cuda()
    s = torch.from_numpy(np.ascontiguousarray(dets[:, 9], dtype=np.float64)).cuda()
    res = core.nms(NMS_HBB, b, s, float(thr_per_group[0]), labels=torch.from_numpy(group.astype(np.int32)).cuda(),
                   thr_per_label=torch.tensor(thr_per_group, dtype=torch.float64, device=b.device), want_mask=False,
                   want_sorted=False, want_score=True, ws_tag="merge")
    kept = res.score_idx.cpu().numpy()
    return kept[np.argsort(group[kept], kind="stable")]


def merge_csv_with_class(data_list, thresh, soft_param=(0.3, 0.6)):
    """:127-156 -- per image, per class NMS over the concatenated submissions."""
    is_dict = isinstance(thresh, dict)
    image_ids = np.unique(data_list[0][:, 0])
    # per image the reference concatenates the submissions in list order; the row order inside a group is
    # (submission, original row), which is what the stable tie-break sees.
    allrows = np.concatenate(data_list)
    rank = np.searchsorted(image_ids, allrows[:, 0])
    rank_c = np.clip(rank, 0, len(image_ids) - 1)
    cls = allrows[:, -1].astype(np.int64)
    valid = (image_ids[rank_c] == allrows[:, 0]) & (cls >= 1) & (cls <= 10)
    rows = allrows[valid]
    if rows.shape[0] == 0:
        raise ValueError("need at least one array to concatenate")  # np.concatenate([]) in the reference
    group = (rank_c[valid] * 10 + (cls[valid] - 1)).astype(np.int32)
    thr = [float(thresh[FAIR1M_1_5_CLASSES[g % 10]]) if is_dict else float(thresh) for g in range(len(image_ids) * 10)]
    return rows[_grouped_nms(rows, group, thr)]


def merge_csv_without_class(data_list, thresh):
    """:159-176 -- per image NMS over all classes."""
    image_ids = np.unique(data_list[0][:, 0])
    allrows = np.concatenate(data_list)
    rank = np.clip(np.searchsorted(image_ids, allrows[:, 0]), 0, len(image_ids) - 1)
    valid = image_ids[rank] == allrows[:, 0]
    rows = allrows[valid]
    if rows.shape[0] == 0:
        raise ValueError("need at least one array to concatenate")
    return rows[_grouped_nms(rows, rank[valid].astype(np.int32), [float(thresh)] * len(image_ids))]
