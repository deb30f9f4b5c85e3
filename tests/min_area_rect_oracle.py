"""numpy/ctypes front-end of min_area_rect_oracle.c (OpenCV's minAreaRect for 4-point polygons, and the mirror's
poly2obb on top of it), plus the seeded quad families the poly2obb tests share.

The C file is compiled with gcc (no FMA contraction) into a temporary directory on first use, so the tests leave the
tree untouched."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(HERE, "min_area_rect_oracle.c")
_lib = None


def lib():
    global _lib
    if _lib is None:
        so = os.path.join(tempfile.mkdtemp(prefix="mar_oracle_"), "libmar_oracle.so")
        subprocess.check_call(["gcc", "-std=c99", "-O2", "-ffp-contract=off", "-fno-fast-math", "-shared", "-fPIC",
                               "-D_DEFAULT_SOURCE", _SRC, "-o", so, "-lm"])
        L = C.CDLL(so)
        L.mar_min_area_rect.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
        L.mar_poly2obb.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
        _lib = L
    return _lib


def _rows(polys):
    return np.ascontiguousarray(np.asarray(polys, np.float64).reshape(-1, 8))


def min_area_rect(polys):
    """(n, 8) -> (n, 5) float32 [cx, cy, w, h, angle in degrees], cv2.minAreaRect of each row as float32 points."""
    p = _rows(polys)
    out = np.zeros((p.shape[0], 5), np.float32)
    lib().mar_min_area_rect(p.ctypes.data, p.shape[0], out.ctypes.data)
    return out


def poly2obb(polys):
    """(n, 8) -> (n, 5) float64 [cx, cy, w, h, theta]: jdet.ops.bbox_transforms.poly2obb."""
    p = _rows(polys)
    out = np.zeros((p.shape[0], 5), np.float64)
    lib().mar_poly2obb(p.ctypes.data, p.shape[0], out.ctypes.data)
    return out


def cv2_min_area_rect(polys):
    """The same as min_area_rect, one cv2.minAreaRect call per row."""
    import cv2
    p = _rows(polys).astype(np.float32).reshape(-1, 4, 2)
    out = [[x, y, w, h, a] for (x, y), (w, h), a in (cv2.minAreaRect(q) for q in p)]
    return np.array(out, np.float32).reshape(-1, 5)


# ---------------------------------------------------------------------------------------------- seeded quad families
def rotated_rects(rng, m, jitter=1.5, smin=2.0, smax=400.0, scene=15000.0):
    """Rotated rectangles in scene coordinates with jittered corners, quantised to 4 decimals as in the CSVs."""
    c = rng.uniform(0, scene, (m, 2))
    w, h = rng.uniform(smin, smax, m), rng.uniform(smin, smax, m)
    t = rng.uniform(-np.pi, np.pi, m)
    ca, sa = np.cos(t)[:, None], np.sin(t)[:, None]
    lx = np.array([-.5, .5, .5, -.5]) * w[:, None]
    ly = np.array([-.5, -.5, .5, .5]) * h[:, None]
    p = np.stack([c[:, :1] + lx * ca - ly * sa, c[:, 1:] + lx * sa + ly * ca], -1)
    return np.round((p + rng.normal(0, jitter, p.shape)).reshape(m, 8), 4)


def near_squares(rng, m):
    return rotated_rects(rng, m, jitter=1e-3, smin=10.0, smax=10.0)


def axis_aligned(rng, m):
    x1, y1 = np.round(rng.uniform(0, 15000, (2, m)), 2)
    w, h = np.round(rng.uniform(0, 300, (2, m)), 1)
    return np.stack([x1, y1, x1 + w, y1, x1 + w, y1 + h, x1, y1 + h], 1)


def integer_grid(rng, m, k=4):
    """Corners on a k x k integer grid: collinear and coincident corners, two- and one-point hulls."""
    return rng.integers(0, k, (m, 8)).astype(np.float64)


def all_orders(polys):
    """Every start vertex in both winding orders: 8 copies of the rows, one block per order."""
    q = np.asarray(polys, np.float64).reshape(-1, 4, 2)
    return np.concatenate([np.roll(r, s, axis=1).reshape(-1, 8) for r in (q, q[:, ::-1]) for s in range(4)])


def families(seed, m):
    """name -> (rows, 8) float64 quads; about 3.2 m rows in all."""
    rng = np.random.default_rng(seed)
    return {
        "rotated": rotated_rects(rng, m),
        "near_square": near_squares(rng, m // 2),
        "axis_aligned": axis_aligned(rng, m // 2),
        "orders": all_orders(rotated_rects(rng, m // 8)),
        "grid": integer_grid(rng, m // 2),
        "grid_orders": all_orders(integer_grid(rng, m // 16, 3)),
    }
