"""numpy front-end of tests/roiaware_oracle.c, the CPU restatement of the roiaware_pool3d ops (TEST INFRASTRUCTURE),
and a float64 rounding-aware classifier of its decisions.  The library is compiled on first use into the temporary
directory (keyed by the source's hash), so the repository tree is never written.

Why a classifier: the GPU evaluates cosf / sinf with the device's routines (at most 2 ulp from the exact value, CUDA
Math API), the oracle with glibc's (at most 1 ulp), so on a rotated box the two may round local_x / local_y differently
and disagree on a pair whose exact coordinate sits within a few ulp of a threshold.  Every other step of the test (the
float subtractions, the z test, the voxel arithmetic of a given local coordinate) is one IEEE operation on both sides.
The classifier calls a decision "decided" when the exact value is farther than a bound E from every threshold, so that
both implementations must agree on it.

The bound on local_x (local_y alike).  With c = cos(-h), s = sin(-h) exact, cosa = c + dc, sina = s + ds,
|dc|, |ds| <= 2 ulp <= 2^-22 (|c|, |s| <= 1, ulp(v) <= 2^-23 |v| for normal v).  The computed
local_x = RN(sx * cosa + RN(sy * -sina)) (or both products rounded) differs from the exact sx * c - sy * s by at most
    |sx| 2^-22 + |sy| 2^-22                       (cosf / sinf)
  + |sy| (1 + 2^-22) 2^-24 [+ |sx| (1 + 2^-22) 2^-24]   (product roundings)
  + |local_x| 2^-24                               (the final rounding; |local_x| <= |sx| + |sy| + the terms above)
  < 2^-21 (|sx| + |sy|),
so E = 2^-20 (|sx| + |sy|) + 2^-140 (a factor 2 to spare, plus room for subnormal products).  The bound holds for
either operand order of the contraction.
A voxel coordinate u = RN(RN(l + half) / res) moves by at most (E + 2^-23 (|l| + |half|)) / |res| + 2^-23 |u| when l
moves by E (again a factor 2 to spare); the index trunc(u) after the unsigned clamp changes only where u crosses -1 or
one of 1 .. n - 1, so the coordinate is decided when the exact u is farther than that from all of them.  res == 0
(a degenerate box) gives +-inf, both mapped to n - 1, or NaN (0 / 0) mapped to 0: decided when the exact l + half is
farther than E from 0."""
from __future__ import annotations

import ctypes
import hashlib
import os
import subprocess
import tempfile

import numpy as np

_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "roiaware_oracle.c")
_lib = None
_f = ctypes.POINTER(ctypes.c_float)
_i = ctypes.POINTER(ctypes.c_int32)
MARGIN_GPU = np.float32(1e-5)
MARGIN_CPU = np.float32(1e-2)


def lib() -> ctypes.CDLL:
    global _lib
    if _lib is None:
        digest = hashlib.sha256(open(_SRC, "rb").read()).hexdigest()[:16]
        path = os.path.join(tempfile.gettempdir(), f"tsmdet_roiaware_oracle_{digest}_{os.getuid()}.so")
        if not os.path.exists(path):
            tmp = f"{path}.{os.getpid()}"
            # -ffp-contract=off: only the explicit fmaf() fuses (the GPU form of the local coordinates)
            subprocess.run(["/usr/bin/gcc", "-O2", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-shared",
                            "-fvisibility=hidden", "-o", tmp, _SRC, "-lm"], check=True, capture_output=True)
            os.replace(tmp, path)
        _lib = ctypes.CDLL(path)
    return _lib


def _f32(a, cols):
    return np.ascontiguousarray(a, dtype=np.float32).reshape(-1, cols)


def points_in_boxes(boxes, pts):
    """boxes (B, T, 7), pts (B, N, 3) -> (B, N) int32: the first box holding each point, else -1 (margin 1e-5)"""
    b, t, n = boxes.shape[0], boxes.shape[1], pts.shape[1]
    bx, px = _f32(boxes, 7), _f32(pts, 3)
    out = np.full((b, n), -1, np.int32)
    lib().rao_points_in_boxes(b, t, n, bx.ctypes.data_as(_f), px.ctypes.data_as(_f), out.ctypes.data_as(_i))
    return out


def points_in_boxes_cpu(boxes, pts):
    """boxes (M, 7), pts (N, 3) -> (M, N) int32 0 / 1 (margin 1e-2, every product rounded)"""
    bx, px = _f32(boxes, 7), _f32(pts, 3)
    out = np.zeros((bx.shape[0], px.shape[0]), np.int32)
    lib().rao_points_in_boxes_cpu(bx.shape[0], px.shape[0], bx.ctypes.data_as(_f), px.ctypes.data_as(_f),
                                  out.ctypes.data_as(_i))
    return out


def forward(rois, pts, feats, out_size, L, method):
    """-> (pts_idx_of_voxels (R,X,Y,Z,L), argmax (R,X,Y,Z,C), pooled (R,X,Y,Z,C)) on zero-filled outputs"""
    X, Y, Z = (out_size,) * 3 if isinstance(out_size, int) else tuple(out_size)
    rx, px = _f32(rois, 7), _f32(pts, 3)
    c = feats.shape[1]
    fx = np.ascontiguousarray(feats, np.float32).reshape(-1, max(c, 1))
    r, p = rx.shape[0], px.shape[0]
    idx = np.zeros((r, X, Y, Z, L), np.int32)
    argmax = np.zeros((r, X, Y, Z, c), np.int32)
    pooled = np.zeros((r, X, Y, Z, c), np.float32)
    lib().rao_forward(r, p, c, X, Y, Z, L, rx.ctypes.data_as(_f), px.ctypes.data_as(_f), fx.ctypes.data_as(_f),
                      argmax.ctypes.data_as(_i), idx.ctypes.data_as(_i), pooled.ctypes.data_as(_f), int(method))
    return idx, argmax, pooled


def boxes_on_points(pts, n, seed):
    """n rotated boxes centred near random points of the cloud (N, 3), so that they hold points"""
    r = np.random.default_rng(seed)
    c = pts[r.integers(0, len(pts), n)] + r.normal(0, 0.3, (n, 3))
    d = r.uniform((1.5, 1.2, 1.2), (4.5, 2.2, 2.0), (n, 3))
    h = r.uniform(-np.pi, np.pi, (n, 1))
    return np.concatenate([c, d, h], 1).astype(np.float32)


def _local(boxes, pts):
    """float32 sx, sy, zz (T, N) as both sides compute them, and the exact local_x / local_y in float64"""
    b = _f32(boxes, 7)[:, None, :]
    p = _f32(pts, 3)[None, :, :]
    with np.errstate(invalid="ignore", over="ignore"):
        sx, sy, zz = p[..., 0] - b[..., 0], p[..., 1] - b[..., 1], p[..., 2] - b[..., 2]  # float32 operations
        h = -b[..., 6].astype(np.float64)
        c, s = np.cos(h), np.sin(h)
        lx = sx.astype(np.float64) * c - sy.astype(np.float64) * s
        ly = sx.astype(np.float64) * s + sy.astype(np.float64) * c
        err = 2.0 ** -20 * (np.abs(sx.astype(np.float64)) + np.abs(sy.astype(np.float64))) + 2.0 ** -140
    return sx, sy, zz, lx, ly, err


def _side(l, thr, err):
    """(surely inside, surely outside) of |l| < thr"""
    with np.errstate(invalid="ignore"):
        a = np.abs(l)
        return a < thr - err, ~(a <= thr + err)  # NaN: surely outside


def _chunked(fn, boxes, pts, *args):
    """fn over slices of the boxes (bounded float64 temporaries), results stacked along the box axis"""
    boxes = _f32(boxes, 7)
    step = max(1, (1 << 21) // max(len(_f32(pts, 3)), 1))
    parts = [fn(boxes[i:i + step], pts, *args) for i in range(0, max(len(boxes), 1), step)]
    if isinstance(parts[0], tuple):
        return tuple(np.concatenate([q[j] for q in parts], 0) for j in range(len(parts[0])))
    return np.concatenate(parts, 0)


def classify(boxes, pts, margin=MARGIN_GPU):
    """boxes (T, 7), pts (N, 3) -> (inside, decided), (T, N) bool each: the exact verdict and whether every rounding of
    local_x / local_y within E gives it"""
    return _chunked(_classify, boxes, pts, margin)


def _classify(boxes, pts, margin):
    b = _f32(boxes, 7).astype(np.float64)[:, None, :]
    _, _, zz, lx, ly, err = _local(boxes, pts)
    with np.errstate(invalid="ignore"):
        zin = np.abs(zz).astype(np.float64) <= b[..., 5] / 2.0  # the same operations on both sides: no rounding doubt
    m = np.float64(np.float32(margin))
    xin, xout = _side(lx, b[..., 3] / 2.0 + m, err)
    yin, yout = _side(ly, b[..., 4] / 2.0 + m, err)
    inside = zin & xin & yin
    decided = ~zin | xout | yout | (xin & yin)
    return inside, decided


def _axis_decided(l, err, half, res, n):
    """is the voxel coordinate of the exact offset l (float64) decided?  half, res float32 (T, 1)"""
    half, res = half.astype(np.float64), res.astype(np.float64)
    with np.errstate(invalid="ignore", divide="ignore", over="ignore"):
        num = l + half
        zero = res == 0
        u = num / np.where(zero, 1.0, res)
        eu = (2 * (err + 2.0 ** -23 * (np.abs(l) + np.abs(half))) / np.abs(np.where(zero, 1.0, res)) +
              2.0 ** -22 * np.abs(u))
        ks = np.array([-1.0] + [float(k) for k in range(1, n)])
        far = np.ones(u.shape, bool)
        for k in ks:  # n <= 256 thresholds
            far &= np.abs(u - k) > eu
        far &= np.isfinite(u)
        return np.where(zero, np.abs(num) > err, far)


def classify_voxels(rois, pts, out_size):
    """rois (R, 7), pts (N, 3) -> (R, N) bool: True where the point's membership AND (when inside) its x / y voxel
    coordinates are decided (the z coordinate is computed identically on both sides)"""
    return _chunked(_classify_voxels, rois, pts, out_size)


def _classify_voxels(rois, pts, out_size):
    X, Y, _ = (out_size,) * 3 if isinstance(out_size, int) else tuple(out_size)
    inside, decided = classify(rois, pts)
    b = _f32(rois, 7)
    _, _, _, lx, ly, err = _local(rois, pts)
    with np.errstate(invalid="ignore", over="ignore"):
        hx, hy = (b[:, 3] / np.float32(2))[:, None], (b[:, 4] / np.float32(2))[:, None]
        rx, ry = (b[:, 3] / np.float32(X))[:, None], (b[:, 4] / np.float32(Y))[:, None]
    vox = _axis_decided(lx, err, hx, rx, X) & _axis_decided(ly, err, hy, ry, Y)
    return decided & (~inside | vox)
