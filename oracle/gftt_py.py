"""Numpy replay of cv::GFTTDetector (goodFeaturesToTrack with the min-eigenvalue score) — TEST INFRASTRUCTURE and the
written spec of the arithmetic rtabmap_b200/csrc/gftt.cuh reproduces bit for bit.

Kp/DetectorStrategy=8 (GFTT/ORB, RTAB-Map's default) detects with cv::GFTTDetector (corelib/src/Features2d.cpp:2083-2178)
and describes with cv::ORB::compute.  OpenCV is a third-party dependency; opencv-python 4.13 is that dependency here and
tests/test_oracle_gftt.py pins this replay to it:

1. cornerMinEigenVal(gray, blockSize, 3), BORDER_REFLECT_101
   * Sobel 8U -> 32F with scale = 1 / (4 * blockSize * 255), k0 = float(scale), k1 = float(2 * scale):
     dx: row pass p[x+1] - p[x-1] (exact integers), column pass fmaf(r[y-1] + r[y+1], k0, r[y] * k1);
     dy: row pass fmaf(R, k0, fmaf(C, k1, L * k0)), except in the columns past the last multiple of 16 (the scalar
         tail of OpenCV's vector loop), where it is (L * k0 + C * k1) + R * k0; column pass r[y+1] - r[y-1];
   * products dx*dx, dx*dy, dy*dy in float;
   * unnormalised blockSize x blockSize box filter: row sums in double (direct, left to right, for 3 and 5 taps; a running
     s += new - old along the whole row for 7), column sums a running double down the whole image:
     s = SUM + new; out = float(s); SUM = s - old;
   * a = cxx * 0.5f, c = cyy * 0.5f, lambda = (a + c) - sqrtf((a - c)^2 + b^2), float, no FMA.
2. goodFeaturesToTrack: maxVal over the mask, THRESH_TOZERO at float(maxVal * qualityLevel), 3x3 dilate; candidates in
   [1, h-2] x [1, w-2], non-zero, equal to the dilated value, inside the mask; sorted by lambda, then address, both
   descending; greedy min-distance pass over a grid of cvRound(minDistance) cells (+-1 cell), stop at maxCorners.
detect_describe() is the whole GFTT/ORB feature block on top of opencv-python itself, as feature2d_py.detect_describe is for ORB.
"""
from __future__ import annotations

from dataclasses import dataclass

import cv2
import numpy as np

from . import feature2d_py as f2d

f32 = np.float32


@dataclass
class GfttParams:
    quality_level: float = 0.001  # GFTT/QualityLevel
    min_distance: float = 7.0     # GFTT/MinDistance
    block_size: int = 3           # GFTT/BlockSize


def detect_describe(image: np.ndarray, depth, K4, p: f2d.OrbParams = f2d.OrbParams(), gftt: GfttParams = GfttParams()):
    """Memory::createSignature's feature block with Kp/DetectorStrategy=8 (GFTT/ORB): cv::GFTTDetector (maxCorners =
    Kp/MaxFeatures, GFTT::generateKeypointsImpl, Features2d.cpp:2148-2178) inside the depth mask, limitKeypoints (a no-op),
    cv::ORB::compute (GFTT_ORB::generateDescriptorsImpl, :2351-2355), generateKeypoints3D.  Same return as
    feature2d_py.detect_describe: (keypoints [n,6] float32 = x,y,size,angle,response,octave; desc [n,32]; xyz [n,3])."""
    gray = cv2.cvtColor(image, cv2.COLOR_BGR2GRAY) if image.ndim == 3 else image
    mask = f2d.depth_mask(depth, p) if (depth is not None and p.depth_as_mask) else None
    kps = cv2.GFTTDetector_create(p.n_features, gftt.quality_level, gftt.min_distance, gftt.block_size).detect(gray, mask)
    kps = f2d.limit_keypoints(kps, p.n_features)
    kps, desc = f2d.make_orb(p).compute(gray, kps)
    if desc is None:
        desc = np.zeros((0, 32), np.uint8)
    xyz = f2d.keypoints_3d(kps, depth, K4, p) if depth is not None else np.full((len(kps), 3), np.nan, np.float32)
    arr = np.array([[k.pt[0], k.pt[1], k.size, k.angle, k.response, k.octave] for k in kps], np.float32).reshape(-1, 6)
    return arr, desc, xyz


def _fma(a, b, c):
    """fmaf(a, b, c) on float32 arrays, rounded once: the float product is exact in double, the double sum is made
    round-to-odd from its exact error (TwoSum), and rounding that to float is then correctly rounded."""
    p = a.astype(np.float64) * b.astype(np.float64)
    q = np.broadcast_to(c, p.shape).astype(np.float64)
    s = p + q
    bb = s - p
    err = (p - (s - bb)) + (q - bb)
    even = (s.view(np.uint64) & np.uint64(1)) == 0
    fix = (err != 0) & even
    s = np.where(fix, np.nextafter(s, s + err), s)
    return s.astype(f32)


def _reflect101(i, n):
    i = np.abs(i)
    return np.where(i >= n, 2 * n - 2 - i, i)


def min_eigen_val(gray: np.ndarray, block_size: int = 3) -> np.ndarray:
    """cv2.cornerMinEigenVal(gray, block_size, 3) bit for bit (float32 [h, w])."""
    assert gray.dtype == np.uint8 and gray.ndim == 2 and block_size in (3, 5, 7)
    h, w = gray.shape
    scale = 1.0 / (4.0 * block_size * 255.0)
    k0, k1 = f32(scale), f32(2.0 * scale)
    xs, ys = np.arange(w), np.arange(h)
    p = gray.astype(np.int32)
    L, C, R = p[:, _reflect101(xs - 1, w)], p, p[:, _reflect101(xs + 1, w)]
    # dx: integer row pass, scaled symmetric column pass
    rx = (R - L).astype(f32)
    up, dn = _reflect101(ys - 1, h), _reflect101(ys + 1, h)
    dx = _fma(rx[up] + rx[dn], np.full_like(rx, k0), rx * k1)
    # dy: scaled row pass (FMA chain in the vector body, plain operations in the scalar tail), antisymmetric column pass
    Lf, Cf, Rf = L.astype(f32), C.astype(f32), R.astype(f32)
    ry = _fma(Rf, np.full_like(Rf, k0), _fma(Cf, np.full_like(Cf, k1), Lf * k0))
    tail = (w // 16) * 16
    if tail < w:
        ry[:, tail:] = (Lf[:, tail:] * k0 + Cf[:, tail:] * k1) + Rf[:, tail:] * k0
    dy = ry[dn] - ry[up]
    cov = [dx * dx, dx * dy, dy * dy]
    r = block_size // 2
    out = []
    for m in cov:
        # row sums in double: direct, left to right, for 3 and 5 taps; a running sum s += new - old for 7
        ext = m[:, _reflect101(np.arange(-r, w + r), w)].astype(np.float64)
        if block_size < 7:
            rs = ext[:, 0:w]
            for d in range(1, block_size):
                rs = rs + ext[:, d:d + w]
        else:
            rs = np.empty((h, w), np.float64)
            s = ext[:, 0]
            for d in range(1, block_size):
                s = s + ext[:, d]
            rs[:, 0] = s
            for x in range(1, w):
                s = s + (ext[:, x + block_size - 1] - ext[:, x - 1])
                rs[:, x] = s
        # running column sum down the whole height
        rows = rs[_reflect101(np.arange(-r, h + r), h)]
        o = np.empty((h, w), f32)
        acc = np.zeros(w, np.float64)
        for k in range(block_size - 1):
            acc = acc + rows[k]
        for y in range(h):
            s = acc + rows[y + block_size - 1]
            o[y] = s.astype(f32)
            acc = s - rows[y]
        out.append(o)
    a = out[0] * f32(0.5)
    b = out[1]
    c = out[2] * f32(0.5)
    t = a - c
    return (a + c) - np.sqrt(t * t + b * b).astype(f32)


def candidates(eig: np.ndarray, quality_level: float, mask=None) -> np.ndarray:
    """goodFeaturesToTrack's candidate list: flat indices sorted by (lambda, address), both descending."""
    h, w = eig.shape
    valid = eig if mask is None else eig[mask != 0]
    max_val = float(valid.max()) if valid.size else 0.0
    thr = f32(max_val * quality_level)
    t = np.where(eig > thr, eig, f32(0))
    pad = np.pad(t, 1, constant_values=-np.inf)
    dil = np.max(np.stack([pad[1 + dy:1 + dy + h, 1 + dx:1 + dx + w] for dy in (-1, 0, 1) for dx in (-1, 0, 1)]), 0)
    ok = (t != 0) & (t == dil)
    ok[0, :] = ok[-1, :] = False
    ok[:, 0] = ok[:, -1] = False
    if mask is not None:
        ok &= mask != 0
    idx = np.flatnonzero(ok)
    lam = t.ravel()[idx]
    order = np.lexsort((-idx, -lam.astype(np.float64)))
    return idx[order]


def select(idx: np.ndarray, w: int, h: int, min_distance: float, max_corners: int) -> np.ndarray:
    """The greedy min-distance pass over the sorted candidates; returns the accepted flat indices in order."""
    if min_distance < 1:
        return idx[:max_corners] if max_corners > 0 else idx
    cell = int(np.round(min_distance))  # cvRound: half to even
    gw, gh = (w + cell - 1) // cell, (h + cell - 1) // cell
    md2 = min_distance * min_distance
    grid = [[] for _ in range(gw * gh)]
    kept = []
    for i in idx.tolist():
        y, x = divmod(i, w)
        xc, yc = x // cell, y // cell
        good = True
        for yy in range(max(yc - 1, 0), min(yc + 1, gh - 1) + 1):
            for xx in range(max(xc - 1, 0), min(xc + 1, gw - 1) + 1):
                for (mx, my) in grid[yy * gw + xx]:
                    if (x - mx) ** 2 + (y - my) ** 2 < md2:
                        good = False
                        break
                if not good:
                    break
            if not good:
                break
        if good:
            grid[yc * gw + xc].append((x, y))
            kept.append(i)
            if max_corners > 0 and len(kept) == max_corners:
                break
    return np.array(kept, np.int64)


def detect(gray: np.ndarray, max_corners: int, quality_level: float = 0.001, min_distance: float = 7.0, block_size: int = 3, mask=None):
    """cv2.GFTTDetector_create(max_corners, quality_level, min_distance, block_size).detect(gray, mask) as an array
    [n, 6] float32 = x, y, size, angle, response, octave (in the detector's order)."""
    h, w = gray.shape
    eig = min_eigen_val(gray, block_size)
    kept = select(candidates(eig, quality_level, mask), w, h, min_distance, max_corners)
    out = np.zeros((len(kept), 6), f32)
    out[:, 0] = kept % w
    out[:, 1] = kept // w
    out[:, 2] = block_size
    out[:, 3] = -1
    out[:, 4] = eig.ravel()[kept]
    return out
