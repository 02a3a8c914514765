"""TEST INFRASTRUCTURE — a restatement of OpenCV's `cv2.line(img, p0, p1, colour, thickness=2)` (LINE_8, shift 0) and
of `cv2.resize(..., INTER_LINEAR)` for uint8 images, in plain Python / numpy.

It is the written specification of ap_pose.cu's rasteriser: tests/test_pose_maps_cpu.py checks it pixel for pixel against
cv2.line's coverage stored in tests/golden/pose_maps.pt, and the kernel follows it step by step.

The thick line, in OpenCV's 16-bit fixed point (XY_SHIFT = 16):
  1. the four corners p0 +- d, p1 -+ d of the quadrilateral around the segment, where d is the unit normal times a
     half-width of 1 px, each component rounded half-to-even (cvRound);
  2. FillConvexPoly of that quadrilateral: the 8-connected outline of its four sides (Line2), then a scanline fill that
     steps a fixed-point x along the left and right edges;
  3. a filled circle of radius 1 (a 5-pixel plus) at each end point;
  4. a zero-length segment gives only the circles.
"""
from __future__ import annotations

import math

import numpy as np

XY_SHIFT = 16
XY_ONE = 1 << XY_SHIFT


def _cdiv(a: int, b: int) -> int:
    """C integer division (truncates toward zero)."""
    q = abs(a) // abs(b)
    return q if (a >= 0) == (b >= 0) else -q


def _clip_line(w: int, h: int, p1, p2):
    """clipLine on the fixed-point image rectangle [0, (w << 16) - 1] x [0, (h << 16) - 1]. Returns None if the segment
    lies outside, else the clipped end points."""
    right, bottom = (w << XY_SHIFT) - 1, (h << XY_SHIFT) - 1
    x1, y1 = p1
    x2, y2 = p2
    c1 = (x1 < 0) + (x1 > right) * 2 + (y1 < 0) * 4 + (y1 > bottom) * 8
    c2 = (x2 < 0) + (x2 > right) * 2 + (y2 < 0) * 4 + (y2 > bottom) * 8
    if (c1 & c2) == 0 and (c1 | c2) != 0:
        if c1 & 12:
            a = 0 if c1 < 8 else bottom
            x1 += int(float(a - y1) * (x2 - x1) / (y2 - y1))
            y1 = a
            c1 = (x1 < 0) + (x1 > right) * 2
        if c2 & 12:
            a = 0 if c2 < 8 else bottom
            x2 += int(float(a - y2) * (x2 - x1) / (y2 - y1))
            y2 = a
            c2 = (x2 < 0) + (x2 > right) * 2
        if (c1 & c2) == 0 and (c1 | c2) != 0:
            if c1:
                a = 0 if c1 == 1 else right
                y1 += int(float(a - x1) * (y2 - y1) / (x2 - x1))
                x1 = a
                c1 = 0
            if c2:
                a = 0 if c2 == 1 else right
                y2 += int(float(a - x2) * (y2 - y1) / (x2 - x1))
                x2 = a
                c2 = 0
    if (c1 | c2) != 0:
        return None
    return (x1, y1), (x2, y2)


def _line2(mask, p1, p2):
    """Line2: the 8-connected line between two fixed-point points."""
    h, w = mask.shape
    clipped = _clip_line(w, h, p1, p2)
    if clipped is None:
        return
    (x1, y1), (x2, y2) = clipped
    dx, dy = x2 - x1, y2 - y1
    ax, ay = abs(dx), abs(dy)

    def put(x, y):
        if 0 <= x < w and 0 <= y < h:
            mask[y, x] = True

    if ax > ay:
        if dx < 0:
            dy = -dy
            x1, x2, y1, y2 = x2, x1, y2, y1
        x_step = XY_ONE
        y_step = _cdiv(dy << XY_SHIFT, ax | 1)
        ecount = (x2 - x1) >> XY_SHIFT
    else:
        if dy < 0:
            dx = -dx
            x1, x2, y1, y2 = x2, x1, y2, y1
        x_step = _cdiv(dx << XY_SHIFT, ay | 1)
        y_step = XY_ONE
        ecount = (y2 - y1) >> XY_SHIFT
    x1 += XY_ONE >> 1
    y1 += XY_ONE >> 1
    put((x2 + (XY_ONE >> 1)) >> XY_SHIFT, (y2 + (XY_ONE >> 1)) >> XY_SHIFT)
    if ax > ay:
        x1 >>= XY_SHIFT
        while ecount >= 0:
            put(x1, y1 >> XY_SHIFT)
            x1 += 1
            y1 += y_step
            ecount -= 1
    else:
        y1 >>= XY_SHIFT
        while ecount >= 0:
            put(x1 >> XY_SHIFT, y1)
            x1 += x_step
            y1 += 1
            ecount -= 1


def _fill_convex_poly(mask, v):
    """FillConvexPoly with shift = XY_SHIFT, LINE_8."""
    h, w = mask.shape
    npts = len(v)
    delta = XY_ONE >> 1
    p0 = v[-1]
    xmin = xmax = v[0][0]
    ymin = ymax = v[0][1]
    imin = 0
    for i, p in enumerate(v):
        if p[1] < ymin:
            ymin, imin = p[1], i
        ymax = max(ymax, p[1])
        xmax = max(xmax, p[0])
        xmin = min(xmin, p[0])
        _line2(mask, p0, p)
        p0 = p
    xmin, xmax = (xmin + delta) >> XY_SHIFT, (xmax + delta) >> XY_SHIFT
    ymin, ymax = (ymin + delta) >> XY_SHIFT, (ymax + delta) >> XY_SHIFT
    if xmax < 0 or ymax < 0 or xmin >= w or ymin >= h:
        return
    ymax = min(ymax, h - 1)
    edge = [dict(idx=imin, di=1, x=-XY_ONE, dx=0, ye=ymin), dict(idx=imin, di=npts - 1, x=-XY_ONE, dx=0, ye=ymin)]
    edges = npts
    y = ymin
    while True:
        for e in edge:
            if y >= e["ye"]:
                idx0 = e["idx"]
                idx = idx0 + e["di"]
                if idx >= npts:
                    idx -= npts
                while True:
                    edges -= 1
                    if edges < 0:
                        break
                    ty = (v[idx][1] + delta) >> XY_SHIFT
                    if ty > y:
                        xs, xe = v[idx0][0], v[idx][0]
                        e["ye"] = ty
                        e["dx"] = _cdiv((xe - xs) * 2 + (ty - y), 2 * (ty - y))
                        e["x"] = xs
                        e["idx"] = idx
                        break
                    idx0 = idx
                    idx += e["di"]
                    if idx >= npts:
                        idx -= npts
        if edges < 0:
            break
        if y >= 0:
            left, right = (1, 0) if edge[0]["x"] > edge[1]["x"] else (0, 1)
            xx1 = (edge[left]["x"] + delta) >> XY_SHIFT
            xx2 = (edge[right]["x"] + delta) >> XY_SHIFT
            if xx2 >= 0 and xx1 < w:
                mask[y, max(xx1, 0):min(xx2, w - 1) + 1] = True
        edge[0]["x"] += edge[0]["dx"]
        edge[1]["x"] += edge[1]["dx"]
        y += 1
        if y > ymax:
            break


def _circle1(mask, cx, cy):
    """Filled circle of radius 1: the pixel and its four neighbours, clipped to the image."""
    h, w = mask.shape
    for x, y in ((cx, cy), (cx - 1, cy), (cx + 1, cy), (cx, cy - 1), (cx, cy + 1)):
        if 0 <= x < w and 0 <= y < h:
            mask[y, x] = True


def corners(x0: int, y0: int, x1: int, y1: int):
    """The thick line's quadrilateral in 16-bit fixed point, or None for a zero-length segment."""
    p0x, p0y, p1x, p1y = x0 << XY_SHIFT, y0 << XY_SHIFT, x1 << XY_SHIFT, y1 << XY_SHIFT
    dx = float(p0x - p1x) / XY_ONE
    dy = float(p1y - p0y) / XY_ONE
    r = dx * dx + dy * dy
    if not abs(r) > np.finfo(np.float64).eps:
        return None
    r = float(XY_ONE) / math.sqrt(r)            # (thickness << 15) for thickness 2, no odd-thickness term
    dpx, dpy = round(dy * r), round(dx * r)     # Python round() is half-to-even, like cvRound
    return [(p0x + dpx, p0y + dpy), (p0x - dpx, p0y - dpy), (p1x - dpx, p1y - dpy), (p1x + dpx, p1y + dpy)]


def thick_line_mask(shape, x0: int, y0: int, x1: int, y1: int) -> np.ndarray:
    """bool [H, W]: the pixels cv2.line(img, (x0, y0), (x1, y1), c, thickness=2) writes."""
    mask = np.zeros(shape, dtype=bool)
    quad = corners(x0, y0, x1, y1)
    if quad is not None:
        _fill_convex_poly(mask, quad)
    _circle1(mask, x0, y0)
    _circle1(mask, x1, y1)
    return mask


# --------------------------------------------------------------------------------------------------------------
# cv2.resize(src, (W, H), interpolation=INTER_LINEAR) for uint8
# --------------------------------------------------------------------------------------------------------------
INTER_BITS = 11
INTER_ONE = 1 << INTER_BITS


def linear_taps(src: int, dst: int):
    """Per output index: (i0, i1, c0, c1). Half-pixel centres with scale 1 / (dst / src), clamped edges, the fraction
    computed in fp32 and each weight rounded half-to-even to 11 bits."""
    scale = 1.0 / (dst / src)
    out = []
    for d in range(dst):
        fx = np.float32((d + 0.5) * scale - 0.5)
        sx = math.floor(fx)
        fx = np.float32(fx - np.float32(sx))
        if sx < 0:
            fx, sx = np.float32(0), 0
        if sx >= src - 1:
            fx, sx = np.float32(0), src - 1
        c0 = int(np.rint(np.float32(np.float32(1) - fx) * np.float32(INTER_ONE)))
        c1 = int(np.rint(fx * np.float32(INTER_ONE)))
        out.append((sx, min(sx + 1, src - 1), c0, c1))
    return out


def resize_linear_u8(img: np.ndarray, W: int, H: int) -> np.ndarray:
    """INTER_LINEAR resize of a uint8 [h, w, C] image to [H, W, C]. Horizontal pass to int32 (weights sum to 2048), then
    OpenCV's vectorised vertical pass: ((r0 >> 4) * b0 >> 16) + ((r1 >> 4) * b1 >> 16), + 2, >> 2. cv2 finishes a row
    whose byte count is not a multiple of its SIMD width with a scalar loop that rounds (sum + 2^21) >> 22 instead; those
    last bytes can differ by 1."""
    h, w = img.shape[:2]
    if (h, w) == (H, W):
        return img.copy()
    tx = np.array(linear_taps(w, W), dtype=np.int64)
    ty = np.array(linear_taps(h, H), dtype=np.int64)
    src = img.astype(np.int64)
    rows = src[:, tx[:, 0]] * tx[:, 2, None] + src[:, tx[:, 1]] * tx[:, 3, None]       # [h, W, C]
    a = ((rows[ty[:, 0]] >> 4) * ty[:, 2, None, None]) >> 16
    b = ((rows[ty[:, 1]] >> 4) * ty[:, 3, None, None]) >> 16
    return np.clip((a + b + 2) >> 2, 0, 255).astype(np.uint8)


def face_mesh_map(keypoints: np.ndarray, groups, W: int, H: int, normed: bool = False) -> np.ndarray:
    """FaceMeshVisualizer.draw_landmarks restated on thick_line_mask / resize_linear_u8: keypoints [N, >= 2];
    groups [(edges, colour)] in drawing order. Returns uint8 [H, W, 3]."""
    kp = np.asarray(keypoints)[:, :2]
    if not normed:
        kp = kp / np.array([W, H], dtype=kp.dtype if kp.dtype == np.float32 else np.float64)
    v = kp.astype(np.float32)
    valid = (v >= 0).all(1) & (v <= 1).all(1)
    px = np.minimum(np.floor(np.where(valid[:, None], v, 0).astype(np.float64) * 512), 511).astype(int)
    img = np.zeros((512, 512, 3), np.uint8)
    for edges, colour in groups:
        cover = np.zeros((512, 512), bool)
        for a, b in edges:
            if valid[a] and valid[b]:
                cover |= thick_line_mask((512, 512), px[a, 0], px[a, 1], px[b, 0], px[b, 1])
        img[cover] = colour
    return resize_linear_u8(img, W, H)
